/* raft_b200.h -- C ABI of the B200-native RAFT forward/update hot path.
 *
 * Drop-in boundary for daigo0927/tf-raft (reference @ 3c85f54).  The reference has no FFI of
 * its own: its boundary is the Python object API of tf_raft/layers/corr.py, tf_raft/layers/update.py
 * and tf_raft/model.py.  Each entry point below replaces the TensorFlow op sequence behind one of
 * those Python calls (cited as file:line); the host-side mirror (tf_raft_b200/) keeps the reference's
 * class / method names and binds these symbols with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every pointer is DEVICE memory, dense row-major, NHWC, float32 unless stated;
 *     coordinates are (x, y) in the last dimension, exactly as in the reference;
 *   - the caller owns every buffer; the library never allocates or frees device memory and
 *     keeps no global mutable state beyond once-initialised function attributes and the
 *     resolved driver entry point for cuTensorMapEncodeTiled;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); nothing
 *     synchronises the device, so a sequence of calls can be captured into a CUDA graph;
 *   - return value: 0 = ok, < 0 = raft_status (argument / shape / workspace error, detected on
 *     the host before anything is launched), > 0 = cudaError_t of a failed launch;
 *   - re-entrant across host threads as long as streams and buffers differ;
 *   - there is NO CPU path: without an sm_100 device every compute entry point returns
 *     RAFT_ERR_NO_DEVICE or the CUDA error.
 */
#ifndef RAFT_B200_H_
#define RAFT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAFT_B200_ABI_VERSION 1
#define RAFT_MAX_LEVELS 8

typedef enum raft_status {
  RAFT_OK = 0,
  RAFT_ERR_BAD_ARG = -1,     /* null pointer, unknown enum value                          */
  RAFT_ERR_BAD_SHAPE = -2,   /* non-positive dims, C not a multiple of 8, level too small */
  RAFT_ERR_WORKSPACE = -3,   /* workspace / prepared-weights buffer too small             */
  RAFT_ERR_NO_DEVICE = -4,   /* no CUDA device of compute capability 10.x                 */
  RAFT_ERR_DRIVER = -5,      /* cuTensorMapEncodeTiled unavailable or rejected a map       */
  RAFT_ERR_UNSUPPORTED = -6  /* valid request this build does not implement               */
} raft_status;

/* Arithmetic of the contraction kernels (correlation GEMM and update-block convolutions).
 * Both are fp32-grade: the final-flow parity gate (<= 1e-3 max-abs) holds for either.
 *   FP32   CUDA-core FFMA, fp32 operands, fp32 accumulate.
 *   F16X2  tcgen05 tensor cores: every fp32 operand v is split into fp16 (hi, lo) with
 *          v ~= hi + lo (22-bit significand), the product is hi*hi + lo*hi + hi*lo
 *          with fp32 accumulation in TMEM (DESIGN.md "Precision").                          */
typedef enum raft_precision { RAFT_PREC_FP32 = 0, RAFT_PREC_F16X2 = 1 } raft_precision;

/* model.py:10-30 (RAFT, BasicUpdateBlock) / model.py:173-188 (SmallRAFT, SmallUpdateBlock). */
typedef enum raft_variant { RAFT_VARIANT_BASIC = 0, RAFT_VARIANT_SMALL = 1 } raft_variant;

const char* raft_b200_strerror(int status);
int raft_b200_abi_version(void);
/* 0 if device `device` can run the kernels (compute capability 10.x), else RAFT_ERR_NO_DEVICE. */
int raft_b200_device_ok(int device);

/* ---------------------------------------------------------------------------------------------
 * CorrBlock  (tf_raft/layers/corr.py:99-162)
 * ------------------------------------------------------------------------------------------- */

/* Bytes of each pyramid level for CorrBlock(fmap1, fmap2, num_levels): level l is
 * (B*h*w, h>>l, w>>l, 1) float32 -- corr.py:108-114 (avg_pool2d 2x2 VALID floors odd dims).   */
int raft_b200_corr_pyramid_sizes(int B, int h, int w, int levels, size_t bytes_per_level[]);

/* Scratch needed by raft_b200_corr_pyramid_build.                                              */
int raft_b200_corr_workspace_bytes(int B, int h, int w, int C, int levels, int precision, size_t* bytes);

/* CorrBlock.__init__ = correlation() + pyramid: corr.py:100-114 and :154-162.
 *   fmap1, fmap2 : (B, h, w, C);  pyr[l] : (B*h*w, h>>l, w>>l, 1), l < levels.
 *   pyr[0][b*h*w + q][y2][x2] = <fmap1[b,q,:], fmap2[b,y2,x2,:]> / sqrt(C); level l is the
 *   2^l x 2^l block mean of level 0 over (y2, x2).                                              */
int raft_b200_corr_pyramid_build(const float* fmap1, const float* fmap2, int B, int h, int w, int C, int levels,
                                 float* const pyr[], void* workspace, size_t workspace_bytes, int precision,
                                 void* stream);

/* CorrBlock.retrieve: corr.py:116-152 with bilinear_sampler corr.py:28-69.
 *   coords : (B, h, w, 2) (x, y);  out : (B, h, w, out_stride) with the first
 *   levels*(2r+1)^2 channels written; channel = level*(2r+1)^2 + a*(2r+1) + b, tap (a, b) has
 *   x-offset a-r and y-offset b-r (corr.py:133-143).  A tap whose clamped x or y coordinate is
 *   an integer is exactly 0 (floor/ceil corners, corr.py:45-60) -- reproduced bit for bit.      */
int raft_b200_corr_lookup(const float* const pyr[], const float* coords, int B, int h, int w, int levels,
                          int radius, float* out, int out_stride, void* stream);

/* Backward of CorrBlock.retrieve for the training step (tf_raft/model.py:133: tape.gradient through corr.py:116-152;
 * the reference does not detach coords1, model.py:102).  grad_out (B, h, w, levels*(2r+1)^2) -> grad_coords (B, h, w, 2)
 * and grad_pyr[l] (same shapes as pyr[l]); both outputs are ACCUMULATED into (zero them first).  TensorFlow gradient
 * rules: floor / ceil / indices carry no gradient, clip_by_value passes it inside [0, dim-1].                        */
int raft_b200_corr_lookup_backward(const float* const pyr[], const float* coords, const float* grad_out, int B, int h, int w,
                                   int levels, int radius, float* grad_coords, float* const grad_pyr[], void* stream);

/* tf.linalg.global_norm over a flat gradient buffer (model.py:135): out[0] = sum g^2 (deterministic two-stage
 * reduction; `partials` holds one float per block, at most npartials blocks are used).                               */
int raft_b200_sumsq(const float* g, size_t n, float* partials, size_t npartials, float* out, void* stream);

/* tf.clip_by_global_norm (model.py:135) + tfa.optimizers.AdamW.apply_gradients (model.py:136, train_chairs.py:87-90)
 * on flat buffers: g' = g * clip / max(sqrt(*sumsq), clip) (clip_norm <= 0: no clipping); var -= wd * var;
 * m = b1 m + (1-b1) g'; v = b2 v + (1-b2) g'^2; var -= lr_t * m / (sqrt(v) + eps), lr_t already bias-corrected.        */
int raft_b200_adamw_step(float* param, const float* grad, float* m, float* v, size_t n, const float* sumsq, float clip_norm,
                         float lr_t, float beta1, float beta2, float epsilon, float weight_decay, void* stream);

/* bilinear_sampler(image, coords): corr.py:28-69.  image (M, H, W, 1), coords (M, P, 2),
 * out (M, P).  Same floor/ceil semantics as above.                                             */
int raft_b200_bilinear_sampler(const float* image, const float* coords, int M, int H, int W, int P, float* out,
                               void* stream);

/* coords_grid(B, h, w): corr.py:72-90 -> (B, h, w, 2), out[b,y,x] = (x, y).                    */
int raft_b200_coords_grid(int B, int h, int w, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Update blocks  (tf_raft/layers/update.py)
 * ------------------------------------------------------------------------------------------- */

/* One keras Conv2D: HWIO kernel (kh, kw, cin, cout) and bias (cout), device pointers.           */
typedef struct raft_conv {
  const float* kernel;
  const float* bias;
  int kh, kw, cin, cout;
} raft_conv;

/* BasicUpdateBlock (update.py:128-141): BasicMotionEncoder :88-95, SepConvGRU :38-49,
 * FlowHead(256) :5-11, mask head :137-141.                                                      */
typedef struct raft_basic_weights {
  raft_conv convc1, convc2, convf1, convf2, conv;                 /* encoder    */
  raft_conv convz1, convr1, convq1, convz2, convr2, convq2;       /* gru        */
  raft_conv fh_conv1, fh_conv2;                                   /* flow_head  */
  raft_conv mask0, mask2;                                         /* mask[0], mask[2] */
} raft_basic_weights;

/* SmallUpdateBlock (update.py:109-116): SmallMotionEncoder :70-76, ConvGRU :17-24, FlowHead(128). */
typedef struct raft_small_weights {
  raft_conv convc1, convf1, convf2, conv;                         /* encoder    */
  raft_conv convz, convr, convq;                                  /* gru        */
  raft_conv fh_conv1, fh_conv2;                                   /* flow_head  */
} raft_small_weights;

/* Weights are re-laid-out once per model (tap-major; for F16X2 also split into scaled fp16
 * hi/lo planes) into a caller-owned device buffer that the update calls then read.              */
int raft_b200_update_prepared_bytes(int variant, int corr_channels, int precision, size_t* bytes);
int raft_b200_update_prepare(int variant, const void* weights /* raft_basic_weights* | raft_small_weights* */,
                             void* prepared, size_t prepared_bytes, int precision, void* stream);

/* Activation scratch for one update call (and for raft_b200_forward_loop) at this shape.        */
int raft_b200_update_workspace_bytes(int variant, int B, int h, int w, int precision, size_t* bytes);

/* BasicUpdateBlock.call([net, inp, corr, flow]) -> (net, 0.25*mask, delta_flow): update.py:143-153.
 *   net, inp : (B,h,w,128); corr : (B,h,w,324); flow : (B,h,w,2)
 *   net_out (B,h,w,128) may alias net; mask (B,h,w,576) may be NULL (skips the mask head);
 *   delta_flow (B,h,w,2).                                                                        */
int raft_b200_update_basic(const void* prepared, const float* net, const float* inp, const float* corr,
                           const float* flow, float* net_out, float* mask_or_null, float* delta_flow, int B,
                           int h, int w, void* workspace, size_t workspace_bytes, int precision, void* stream);

/* SmallUpdateBlock.call -> (net, None, delta_flow): update.py:118-125.
 *   net (B,h,w,96), inp (B,h,w,64), corr (B,h,w,196), flow (B,h,w,2).                            */
int raft_b200_update_small(const void* prepared, const float* net, const float* inp, const float* corr,
                           const float* flow, float* net_out, float* delta_flow, int B, int h, int w,
                           void* workspace, size_t workspace_bytes, int precision, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Encoders  (tf_raft/layers/extractor.py) -- SURVEY.md section 8(f) rank 1
 * ------------------------------------------------------------------------------------------- */

/* One normalisation layer: tfa InstanceNormalization (gamma, beta) or keras BatchNormalization (+ moving
 * statistics); all (C,) device pointers; NULL members for norm_type NONE.  eps = 1e-3 (extractor.py:6-16).   */
typedef struct raft_norm {
  const float* gamma;
  const float* beta;
  const float* moving_mean;
  const float* moving_variance;
} raft_norm;

/* ResBlock (extractor.py:19-49); downsample.kernel == NULL when strides == 1.                              */
typedef struct raft_resblock {
  raft_conv conv1, conv2;
  raft_norm norm1, norm2;
  raft_conv downsample;
  raft_norm downsample_norm;
} raft_resblock;

/* BasicEncoder / SmallEncoder (extractor.py:88-175): conv1 7x7 s2, norm1, layer1..3 (2 ResBlocks each,
 * in order layer1.0, layer1.1, layer2.0, ...), conv2 1x1.                                                   */
typedef struct raft_encoder_weights {
  raft_conv conv1;
  raft_norm norm1;
  raft_resblock block[6];
  raft_conv conv2;
} raft_encoder_weights;

typedef enum raft_norm_type { RAFT_NORM_NONE = 0, RAFT_NORM_INSTANCE = 1, RAFT_NORM_BATCH = 2 } raft_norm_type;

int raft_b200_encoder_prepared_bytes(int variant, int out_dim, size_t* bytes);
int raft_b200_encoder_prepare(int variant, int norm_type, int out_dim, const raft_encoder_weights* weights,
                              void* prepared, size_t prepared_bytes, void* stream);
int raft_b200_encoder_workspace_bytes(int variant, int N, int H, int W, size_t* bytes);

/* BasicEncoder.call / SmallEncoder.call (extractor.py:113-130 / 158-175) on N images.
 *   images : (N, H, W, 3); image_norm != 0: values are 0..255 and the 2*(x/255)-1 of model.py:70-71 is
 *            fused into the first load; image_norm == 0: already normalised (the encoder layer on its own)
 *   out    : (N, ceil(H/8), ceil(W/8), out_dim)
 *   training != 0 selects batch statistics for RAFT_NORM_BATCH (moving statistics are not updated here).   */
int raft_b200_encoder_forward(int variant, int norm_type, int out_dim, const void* prepared, const float* images,
                              int N, int H, int W, int training, int image_norm, float* out, void* workspace,
                              size_t workspace_bytes, void* stream);

/* model.py:84-86: net = tanh(cnet[..., :hidden]), inp = relu(cnet[..., hidden:]).                          */
int raft_b200_context_split(const float* cnet, int npix, int hidden, int context, float* net, float* inp,
                            void* stream);

/* One keras Conv2D(cout, (kh, kw), 1, 'same') + optional activation on its own (fp32 FFMA path): the building block
 * behind the stand-alone FlowHead / ConvGRU / SepConvGRU / *MotionEncoder layers of update.py:5-106 when they are
 * used outside the fused update block.  x (B,H,W,cin), kernel HWIO, out (B,H,W,out_stride) written at channel out_c0.
 * act: 0 none, 1 relu, 2 sigmoid, 3 tanh.                                                                        */
int raft_b200_conv2d(const float* x, const float* kernel, const float* bias, int B, int H, int W, int cin, int kh,
                     int kw, int cout, int act, float* out, int out_stride, int out_c0, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Model loop  (tf_raft/model.py)
 * ------------------------------------------------------------------------------------------- */

/* RAFT.upsample_flow(flow, mask): model.py:39-66.  flow (B,h,w,2), mask (B,h,w,576) with channel
 * (by*8+bx)*9 + ky*3+kx -> out (B,8h,8w,2): softmax over the 9 taps of the zero-padded 3x3
 * neighbourhood of 8*flow, depth_to_space(8).                                                    */
int raft_b200_upsample_convex(const float* flow, const float* mask, int B, int h, int w, float* out, void* stream);

/* upflow8(flow): corr.py:93-96 = 8 * bilinear resize with half-pixel centres.                    */
int raft_b200_upflow8(const float* flow, int B, int h, int w, float* out, void* stream);

/* The iteration loop of RAFT.call / SmallRAFT.call: model.py:93-106 / :212-224.
 *   for i < iters:  corr = retrieve(coords1); flow = coords1 - coords0;
 *                   net, mask, delta = update_block([net, inp, corr, flow]);
 *                   coords1 += delta;  flow_up[i] = upsample(coords1 - coords0, mask)
 *   pyr          : the CorrBlock pyramid (levels entries)
 *   net          : (B,h,w,hidden) in/out -- the tanh() half of cnet's output on entry
 *   inp          : (B,h,w,context)       -- the relu() half
 *   coords1      : (B,h,w,2) in/out; the starting point: coords_grid(B,h,w) (model.py:89), or
 *                  coords_grid + an initial flow to warm-start the loop (flow is always taken as
 *                  coords1 - the pixel grid, whatever coords1 held on entry)
 *   flow_up      : iters pointers to (B,8h,8w,2) outputs; entries may be NULL to skip that
 *                  iteration's upsampling (predict_step keeps only the last, model.py:166);
 *                  for BASIC a skipped iteration also skips the mask head.                        */
int raft_b200_forward_loop(int variant, const void* prepared, const float* const pyr[], int levels, int radius,
                           float* net, const float* inp, float* coords1, float* const flow_up[], int iters,
                           int B, int h, int w, void* workspace, size_t workspace_bytes, int precision,
                           void* stream);

/* Warm start for the next pair of a video (the original RAFT's forward_interpolate).
 * flow (B,h,w,2). Sample (x,y) lands at px = x + fx, py = y + fy (in fp64). It is kept iff
 * 0 < px < w and 0 < py < h, strictly; NaN is never kept. For every grid point q = (qx,qy):
 *   out(q) = flow of the kept sample with the least d2 = ((qx-x)-fx)^2 + ((qy-y)-fy)^2,
 *   evaluated in fp64 op by op (no FMA contraction). Ties go to the lowest row-major index.
 *   If an image keeps no sample, out = 0 for that image.
 * out_coords = 1 writes coords_grid + that flow instead (fp32 add): the coords1 the forward loop starts from.
 * out must not overlap flow (RAFT_ERR_BAD_ARG); B <= 65535, h*w <= 2^30. Cost is O((h*w)^2) per image.
 * No workspace, no allocation, no sync.                                                           */
int raft_b200_forward_interpolate(const float* flow, int B, int h, int w, int out_coords, float* out, void* stream);

/* Number of kernels the most recent call on this host thread launched (bench.py's gpu_launches). */
long long raft_b200_launch_count(void);
void raft_b200_launch_count_reset(void);
/* Profiling aid for bench.py's roofline objects: while enabled, raft_b200_forward_loop (F16X2, <= 64 iterations, not
 * under CUDA-graph capture) records CUDA events on its stream around the lookup and around the update-block kernel(s)
 * of every iteration; _read waits for the last one and returns the summed durations of the most recent call.      */
void raft_b200_profile_loop(int enable);
int raft_b200_profile_read(float* lookup_ms, float* update_ms, int* iterations);
/* Profiling aid: the next update-block launches of tensor-core layer `tc_layer` (-1 = off; 2000 = the correlation kernel) write clock64 stamps of
 * CTA 0 into `device_buf_2048` (4 x 512 int64: slot free / data landed / group retired / group drained).        */
void raft_b200_debug_timeline(int tc_layer, long long* device_buf_2048);

#ifdef __cplusplus
}
#endif
#endif /* RAFT_B200_H_ */
