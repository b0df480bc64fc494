/* atvs.h - C ABI of libatvs.so: the B200 (sm_100a) implementation of the A-TVSNet
 * inference hot path.
 *
 * The reference (daiszh/A-TVSNet) has no FFI layer: its boundary for this path is a set
 * of Python functions building TensorFlow-1.5 graph ops.  Each entry point below states
 * which reference function (file:line under /root/reference) it replaces; the Python
 * package `a-tvsnet_b200` re-exposes them under the reference's own names and tensor
 * layouts (see INTEGRATION.md for the binding a maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name
 *     ends in `_host`; the caller owns every buffer, including workspaces;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), which must belong to the calling
 *     thread's current device: every launch and query applies to that device;
 *   - state: the library holds, per device (ordinals 0..63), the fp16 saturation counter, the concurrency hint of
 *     atvs_set_concurrency, the SM count, the shared-memory attribute of each tensor-core kernel (set race-free from
 *     any host thread) and the occupancy of each grid-stride kernel, each set up by the first call on that device
 *     that needs it; such a call on a device beyond 63 fails with ATVS_E_UNSUP.  Per process it holds only the
 *     launch counter and host constants (the CRC-32C table, the driver's tensor-map encoder);
 *   - return value: 0 = ok, >0 = cudaError_t / CUresult of the failing call,
 *     <0 = argument error (ATVS_E_*); atvs_last_error() returns a thread-local message;
 *   - activations are channels-last (B,D,H,W,C), exactly the reference's NDHWC layout;
 *   - dtype codes: ATVS_F32 = 0, ATVS_BF16 = 1, ATVS_F16 = 2.  The tensor-core path keeps activations and weights
 *     in ONE 16-bit format, ATVS_F16 (default: 11 significant bits; BN-normalised activations are bounded, so the
 *     5-bit exponent is enough; conversions saturate) or ATVS_BF16; both run tcgen05.mma.kind::f16 at the same rate.
 */
#ifndef ATVS_H_
#define ATVS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ATVS_F32  0
#define ATVS_BF16 1
#define ATVS_F16  2

#define ATVS_E_SHAPE  (-1)   /* bad shape / alignment                     */
#define ATVS_E_DTYPE  (-2)   /* unsupported dtype code                    */
#define ATVS_E_DIV8   (-3)   /* a dimension that must be even / div by 8  */
#define ATVS_E_NULL   (-4)   /* required pointer is NULL                  */
#define ATVS_E_UNSUP  (-5)   /* unsupported configuration                 */

typedef void* atvs_stream_t;     /* cudaStream_t */

int         atvs_version(void);                 /* major*10000 + minor*100 + patch        */
const char* atvs_last_error(void);              /* thread-local, never NULL               */
int         atvs_device_sm_count(void);         /* SMs of the current device (148 on B200) */
long long   atvs_launch_count(void);            /* kernels launched by this library so far  */
/* host helper: CRC-32C (Castagnoli) of n HOST bytes continuing from `crc` (0 to start); the tensor checksums of a
 * TensorFlow V2 checkpoint, example.py:121-125 (ckpt.py verifies every tensor with it)                          */
unsigned    atvs_crc32c(const void* data_host, size_t n, unsigned crc);
/* number of fp16 raw-output rows (8..32 channels of one voxel) that held a value beyond +-65504 and were clamped by
 * the tensor-path epilogues on the current device since the last reset; synchronises the device; -1 on error.  A
 * non-zero count means the checkpoint's feature scale does not fit fp16 raw storage: rerun with fp32 raw outputs. */
long long   atvs_saturation_count(int reset);
/* Scheduling hint (no effect on results): how many independent regularisation passes the caller runs side by side on
 * its own streams of the current device - the 2*(N-1) passes of example.py:144-158 are independent.  The persistent
 * tensor kernels launch all resident CTAs when a pass has the GPU to itself (n = 1, the default) and fewer, longer
 * CTAs when n passes share the SMs.  Each device keeps its own hint.  Returns 0.                                */
int         atvs_set_concurrency(int n);

/* ---- get_homographies ------------------------------------------- homography_warping.py:179-227
 * left_cam/right_cam (B,2,4,4) f32, depth_start/depth_interval (B) f32 -> out (B,D,3,3) f32.
 * inverse_depth mirrors FLAGS.inverse_depth (homography_warping.py:215).  fp32, fixed op order
 * (no FMA contraction), bit-identical to oracle/homography_warping.py:get_homographies.       */
int atvs_get_homographies(const float* left_cam, const float* right_cam, int B, int D,
                          const float* depth_start, const float* depth_interval,
                          int inverse_depth, float* out, atvs_stream_t stream);

/* ---- homography_warping (+ interpolate) -------------------- homography_warping.py:230-271, 31-104
 * image (B,H,W,C) f32, homography (B,3,3) f32 -> out (B,H,W,C) f32, mask (B,H,W) u8 or NULL.
 * method: 0 = bilinear, 1 = nearest.  C must be a multiple of 4 or equal to 1.                */
int atvs_homography_warping(const float* image, const float* homography, int B, int H, int W,
                            int C, int method, float* out, uint8_t* mask, atvs_stream_t stream);

/* ---- homography_warping_by_depth ------------------------------ homography_warping.py:108-176
 * depth_image (B,H,W) f32 (inverse depth when inverse_depth != 0).                            */
int atvs_homography_warping_by_depth(const float* image, const float* left_cam,
                                     const float* right_cam, const float* depth_image, int B,
                                     int H, int W, int C, int method, int inverse_depth,
                                     float* out, uint8_t* mask, atvs_stream_t stream);

/* ---- build_cost_volume (fused warp + two-view cost) ------------------------- model.py:157-200
 * ref/view feature (B,h,w,F) f32, homographies (B,D,3,3) f32 (view), ref_homographies
 * (B,D,3,3) or NULL (warp_ref=False: the reference half is tile(ref, D)).
 * mode 0 CONCAT      -> out (B,D,h,w,2F)  = [ref | warp(view)]           (reference layout)
 * mode 1 WARPED_ONLY -> out (B,D,h,w,F)   = warp(view)
 * mode 2 L1_MASKED   -> out (B,D,h,w,F)   = |warp(view) - ref| * valid    (model.py:272-280)
 * out_dtype ATVS_F32 | ATVS_BF16 | ATVS_F16.  F must be a multiple of 4 (8 for 16-bit volumes).  Warped feature
 * volumes are never materialised: each plane's slice is streamed straight to `out`.           */
int atvs_build_cost_volume(const float* ref_feature, const float* view_feature,
                           const float* homographies, const float* ref_homographies, int B,
                           int D, int h, int w, int F, int mode, int out_dtype, void* out,
                           atvs_stream_t stream);
/* The same with the source (view) feature map already 16-bit in the volume's own format `dtype` (ATVS_F16 | ATVS_BF16),
 * e.g. converted once per frame for all the passes that warp it: one launch, no scratch (atvs_build_cost_volume makes
 * that copy itself on every call).  ref_feature stays f32 (unused in mode 1).  F in {8, 16, 32, 64, 128}.        */
int atvs_build_cost_volume_src16(const float* ref_feature, const void* view_feature16,
                                 const float* homographies, int B, int D, int h, int w, int F,
                                 int mode, int dtype, void* out, atvs_stream_t stream);

/* ---- 3-D convolution primitives ------------------ network.py:142-215 (conv, conv_bn), 511-550
 * x (B,D,H,W,Cin) dtype `dtype`; kernel in TF layout: conv [3,3,3,Cin,Cout] f32, transposed
 * conv [3,3,3,Cout,Cin] f32; stride 1|2 for conv (TF SAME padding), 2 for the transposed conv
 * (TF SAME: out = 2*in, out[2i+k] += in[i]*w[k]).  No bias.  raw_out (B,Do,Ho,Wo,Cout) f32 is
 * the PRE-batch-norm result.  stats (2*Cout doubles: sum, sum of squares; caller zeroes it)
 * receives the per-channel moments of raw_out when not NULL (batch-statistics BN, F4).
 * atvs_conv3d_fp32: CUDA-core fp32 parity path.  atvs_conv3d_tc: tcgen05/TMEM implicit GEMM,
 * 16-bit operands (x_dtype = ATVS_F16 | ATVS_BF16, the same format as the packed weights), fp32 accumulation;
 * `wpacked` comes from atvs_pack_conv_weights_tc.  The tensor path writes raw_out as raw_dtype = ATVS_F32 or
 * ATVS_F16 (saturated; for layers whose raw output only feeds atvs_bn_relu_add*: the moments still come from the
 * fp32 accumulators, the BN pass rounds to 16 bits right after, and the bytes written here and read there are
 * halved).                                                                                          */
int atvs_conv3d_fp32(const float* x, const float* kernel, int B, int D, int H, int W, int Cin,
                     int Cout, int stride, int transposed, float* raw_out, double* stats,
                     atvs_stream_t stream);

size_t atvs_packed_weight_bytes(int Cin, int Cout, int transposed);
int atvs_pack_conv_weights_tc(const float* kernel, int Cin, int Cout, int transposed, int dtype,
                              void* wpacked, atvs_stream_t stream);
int atvs_conv3d_tc(const void* x16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin,
                   int Cout, int stride, int transposed, void* raw_out, int raw_dtype, double* stats,
                   atvs_stream_t stream);
/* same convolution plus a depth-invariant term: raw_out[b,z,y,x,:] += plane_bias[b,c(z),y,x,:] with
 * c(z) = 0 for the first output plane, 2 for the last, 1 otherwise; plane_bias (B,3,Ho,Wo,Cout) f32.
 * Used for the first CRM layers: the cost volume of model.py:186-195 is [tile(ref, D) | warped], so the
 * reference half of the convolution is a 2-D result shared by all interior planes (computed once by
 * running this same primitive on a 3-plane (4 for stride 2) tile of the reference feature).         */
int atvs_conv3d_tc_bias(const void* x16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin,
                        int Cout, int stride, const float* plane_bias, void* raw_out, int raw_dtype,
                        double* stats, atvs_stream_t stream);

/* ---- batch-norm (batch statistics) + ReLU + skip adds ------ network.py:206-215, 541-550, 696
 * y = relu((raw - mean) * rsqrt(var + eps)) with mean/var from `stats` over `count` voxels
 * (biased variance); out_plain = y (may be NULL); out_sum = y + skip1 + skip2 (NULL skips are
 * omitted; may be NULL).  act_dtype is the dtype of skips and outputs, raw_dtype (ATVS_F32 | ATVS_F16)
 * that of the raw tensor(s).  n = count * C.                                                     */
int atvs_bn_relu_add(const void* raw, int raw_dtype, const double* stats, long long count, int C, float eps,
                     int relu, const void* skip1, const void* skip2, void* out_plain,
                     void* out_sum, int act_dtype, atvs_stream_t stream);

/* `add` of TWO freshly convolved layers (network.py:696 over two conv_bn / deconv_bn outputs, e.g.
 * conv_b1_0_0 = add(conv_b0_6_0, conv_b0_0_1), cnn_wrapper/atvsnet.py:128-131):
 * out_sum = relu(bn(raw_a)) + relu(bn(raw_b)) + skip, each raw tensor with its own batch statistics;
 * out_plain_a = relu(bn(raw_a)) (may be NULL).  Saves writing and re-reading the normalised raw_b.  */
int atvs_bn_relu_add_pair(const void* raw_a, const double* stats_a, const void* raw_b,
                          const double* stats_b, int raw_dtype, long long count, int C, float eps, int relu,
                          const void* skip, void* out_plain_a, void* out_sum, int act_dtype,
                          atvs_stream_t stream);

/* ---- elementwise helpers (dtype plumbing for NDHWC volumes) */
int atvs_cast(const void* src, int src_dtype, void* dst, int dst_dtype, long long n,
              atvs_stream_t stream);
/* fp32 rows (rows, C) -> 16-bit rows (rows, Cpad), channels C..Cpad-1 zero: the input groups of the refinement U-Net
 * (48 / 19 / 1 channels, model.py:328-333) in the tensor-core kernels' channel counts.  Cpad % 8 == 0.                  */
int atvs_pad_cast(const float* x, long long rows, int C, int Cpad, void* out, int out_dtype /* ATVS_F16 | ATVS_BF16 */,
                  atvs_stream_t stream);
int atvs_add(const void* a, const void* b, void* out, int dtype, long long n, atvs_stream_t stream);

/* ---- attention aggregation (AAM) ------------------------------- network.py:282-351, 379-408
 * act (N,V,2C) `dtype`: per view n the pair [relu(conv(x_n,W_unique)) | relu(conv(x_n,W_shared))]
 * (from the conv primitives with W_unique||W_shared concatenated on Cout);
 * x (N,V,C) `dtype`: the per-view cost volumes.  score = softmax_n((u_n - s_n) + sum_m s_m),
 * out (V,C) f32 = sum_n score_n * x_n.  When num_den != NULL the kernel instead writes the
 * un-normalised partials [sum_n e^{l_n - gmax} x_n | sum_n e^{l_n - gmax}] (V,2C) f32 with
 * l_n = u_n - s_n and gmax (V,C) f32 supplied by the caller (multi-GPU source-view sharding);
 * atvs_attention_local_max produces the per-rank max, atvs_attention_finish divides.          */
int atvs_attention_combine(const void* act, const void* x, int N, long long V, int C, int dtype,
                           float* out, atvs_stream_t stream);
int atvs_attention_local_max(const void* act, int N, long long V, int C, int dtype, float* lmax,
                             atvs_stream_t stream);
int atvs_attention_partial(const void* act, const void* x, int N, long long V, int C, int dtype,
                           const float* gmax, float* num_den, atvs_stream_t stream);
int atvs_attention_finish(const float* num_den, long long V, int C, float* out,
                          atvs_stream_t stream);
/* the same three operations (mode 0 = combine, 1 = local max, 2 = partial) on the RAW fp32 output
 * (N,V,2C) of the attention convolution: relu (network.py:323-344) is applied while loading, the
 * activations are never stored.  C % 8 == 0.                                                      */
int atvs_attention_raw(const void* act_raw, int act_dtype /* ATVS_F32 | ATVS_F16 */,
                       const void* const* x_views /* HOST array of N device pointers, each (V,C) x_dtype */, int N,
                       long long V, int C, int x_dtype, int mode, const float* gmax, float* out,
                       atvs_stream_t stream);

/* The whole module in ONE kernel (csrc/conv_attn_ring.cu): the 8 -> 16 attention convolution [W_unique | W_shared] of
 * every view, ReLU, softmax over the views and the weighted sum, with the logits kept in TMEM (never in HBM).
 * network.py:282-351 + :379-408 for C = 8 channels and 2..8 views of one 16-bit dtype.
 * x_views: HOST array of N device pointers, each (B,D,H,W,8) x_dtype; wpacked: atvs_pack_conv_weights_tc(Cin 8,
 * Cout 16, not transposed) of the concatenated kernel, same dtype; out (B,D,H,W,8) fp32.  D >= 3, H, W >= 8.      */
int atvs_attention_fused(const void* const* x_views, int N, int x_dtype /* ATVS_BF16 | ATVS_F16 */, const void* wpacked,
                         int B, int D, int H, int W, int C, float* out, atvs_stream_t stream);

/* ---- 2-D feature extraction module (FEM, ResNetDS2SPP) --- cnn_wrapper/atvsnet.py:254-292, network.py:142-215, 552-671
 * fp32 NHWC CUDA-core parity path of SURVEY.md 8(f) row N1; atvs_conv2d_tc below is the tensor-core path of its
 * stride-1 convolutions.
 * atvs_conv2d_fp32: kernel [k,k,Cin,Cout] (TF layout), k = 1 | 3, stride, dilation `rate`, explicit zero padding
 *   pad_top / pad_left (bottom / right follow from Ho, Wo): TF 'SAME' and the bottleneck's pad + 'VALID'
 *   (network.py:589-595) are both expressed this way; out (B,Ho,Wo,Cout) = [relu](conv + bias), bias may be NULL.
 * atvs_channel_moments: stats[0..C) += sum, stats[C..2C) += sum of squares over `count` rows (caller zeroes stats).
 * atvs_bn2d_apply: (x - mean) * rsqrt(var + eps) [+ beta[c]] [relu], batch statistics from stats / count
 *   (tf.layers.batch_normalization(center=False) -> beta NULL; slim.batch_norm -> beta).
 * atvs_avg_pool_same: tf.layers.average_pooling2d 'SAME', mean over the valid elements; out (B,ceil(H/s),ceil(W/s),C).
 * atvs_resize_bilinear_align: tf.image.resize_images(bilinear, align_corners=True), TF's lerp order.            */
int atvs_conv2d_fp32(const float* x, const float* kernel, const float* bias, int B, int H, int W, int Cin,
                     int Cout, int ksize, int stride, int rate, int pad_top, int pad_left, int Ho, int Wo,
                     int relu, float* out, atvs_stream_t stream);
int atvs_channel_moments(const float* x, long long count, int C, double* stats, atvs_stream_t stream);
int atvs_bn2d_apply(const float* x, const double* stats, const float* beta, long long count, int C, float eps,
                    int relu, void* out, int out_dtype /* ATVS_F32 | ATVS_F16 (saturated) */, atvs_stream_t stream);
int atvs_avg_pool_same(const float* x, int B, int H, int W, int C, int ksize, int stride, float* out,
                       atvs_stream_t stream);
int atvs_resize_bilinear_align(const float* x, int B, int H, int W, int C, int Ho, int Wo, float* out,
                               atvs_stream_t stream);

/* ---- 2-D convolutions of the FEM on tcgen05 -------------- network.py:142-215 (conv, conv_bn), 570-599 (slim.conv2d)
 * stride 1, k = 1 | 3, dilation `rate`, TF 'SAME' padding, as the D = 1 case of the 3-D implicit-GEMM kernel: x16
 * (B,H,W,Cin) ATVS_F16 | ATVS_BF16 with Cin = 32 or a multiple of 64 (read through one TMA map per 64-channel chunk);
 * wpacked from atvs_pack_conv2d_weights_tc (kernel [k,k,Cin,Cout] f32, atvs_packed_weight2d_bytes bytes, Cout <= 256);
 * out (B,H,W,Cout) = [relu](conv + bias[c]) stored as out_dtype = ATVS_F32 | ATVS_F16 (saturated); bias may be NULL;
 * stats (2*Cout doubles, caller zeroes) receives the per-channel moments of the stored value's fp32 source when not
 * NULL (the conv_bn layers).  Stride-2 / 3-channel layers stay on atvs_conv2d_fp32.                              */
size_t atvs_packed_weight2d_bytes(int Cin, int Cout, int ksize);
int atvs_pack_conv2d_weights_tc(const float* kernel, int Cin, int Cout, int ksize, int dtype, void* wpacked,
                                atvs_stream_t stream);
int atvs_conv2d_tc(const void* x16, int x_dtype, const void* wpacked, const float* bias, int B, int H, int W, int Cin,
                   int Cout, int ksize, int rate, int relu, void* out, int out_dtype, double* stats,
                   atvs_stream_t stream);

/* ---- refinement-stage geometry (stage III, SURVEY.md 8(f) N2) ----- homography_warping.py:275-387, model.py:269-337
 * fp32 first path.  atvs_transform_depth: depth (B,H,W) of the left view re-expressed in the right camera, on the left
 *   pixel grid (inverse depth in and out when inverse_depth).
 * atvs_refine_geo_group: (B,D,H,W,C+3) = [ |d_ref - v|/di/D | (|bilinear warp(d_view_trans, H_d) - v|/di/D)*mask x C |
 *   |wg - d_ref|*wg_mask | d_ref ], v = start + d*interval; wg / wg_mask = nearest by-depth warp of d_view_trans
 *   (atvs_homography_warping_by_depth); the C-fold repetition is the reference's tiled mask (C = 16 -> 19 channels).
 * atvs_refine_photo_group: (B,D,H,W,3C) = [cost_photo (B,D,H,W,C) from atvs_build_cost_volume(L1_MASKED) |
 *   |warped_feature - ref_feature|*mask tiled over D | ref_feature tiled over D].
 * atvs_visual_hull: (B,D,H,W) for view_num = 2: ([ref>0][ref beyond plane] + [w>0][w beyond plane]) / 2 with w the
 *   nearest homography warp of trans_depth by H_d.                                                            */
int atvs_transform_depth(const float* depth, const float* left_cam, const float* right_cam, int B, int H, int W,
                         int inverse_depth, float* out, atvs_stream_t stream);
int atvs_refine_geo_group(const float* d_ref, const float* d_view_trans, const float* homographies, const float* wg,
                          const uint8_t* wg_mask, const float* depth_start, const float* depth_interval, int B, int D,
                          int H, int W, int C, float* out, atvs_stream_t stream);
int atvs_refine_photo_group(const float* cost_photo, const float* warped_feature, const uint8_t* mask,
                            const float* ref_feature, int B, int D, int H, int W, int C, float* out,
                            atvs_stream_t stream);
int atvs_visual_hull(const float* ref_depth, const float* trans_depth, const float* homographies,
                     const float* depth_start, const float* depth_interval, int B, int D, int H, int W, int view_num,
                     int inverse_depth, float* out, atvs_stream_t stream);

/* ---- depth-map fusion (post-processing, SURVEY.md 8(f) N4) ------ fusibile/fusibile.cu:138-277 (kernel), :279-325 (scan)
 * normals_depths (N,H,W,4) f32 = (nx, ny, nz, depth) per view (depth_fusion.py:93-112 writes normals (1,1,1)/sqrt(3) where
 * depth > 0), images (N,H,W,4) f32 colour or NULL; cameras as the reference's Camera_cu holds them: cam_P (N,3,4) =
 * (K E)[0:3], cam_Minv (N,3,3) = P[:, :3]^-1, cam_C (N,3) centre, cam_f (N) = K[0,0].  A reference pixel becomes a point
 * when at least num_consistent other views agree: |disp - disp'| / disp < depth_thresh on the projected depth and the
 * angle between the normals < normal_thresh (radians).  All reference cameras in one call; the points are compacted on the
 * device in the reference's order (camera-major, row-major; zero coordinates dropped): out_coord / out_normal
 * (capacity,3), out_texture (capacity,4) or NULL, *out_count (device) = number of points found (may exceed capacity:
 * only the first `capacity` are written).  workspace: atvs_fuse_workspace_bytes(N,H,W) device bytes, 256-byte aligned. */
size_t atvs_fuse_workspace_bytes(int N, int H, int W);
int atvs_fuse_depth_maps(const float* normals_depths, const float* images, const float* cam_P, const float* cam_Minv,
                         const float* cam_C, const float* cam_f, int N, int H, int W, float depth_thresh,
                         float normal_thresh, int num_consistent, int save_texture, void* workspace, long long capacity,
                         float* out_coord, float* out_normal, float* out_texture, long long* out_count,
                         atvs_stream_t stream);

/* ---- prob2depth / get_propability_map / prob2depth_upsample -------- model.py:80-129, 13-76
 * prob_volume (B,D,H,W) f32 logits; softmax over D of -logit, expectation against
 * linspace(start, start+(D-1)*interval, D) -> depth (B,H*up,W*up) f32; prob_map (same shape,
 * sum of the 4 probabilities around the estimate) or NULL.  up = 1, or 4 for the fused
 * bilinear (align_corners) x4 logit upsample of model.py:68-76 (never materialised).          */
int atvs_prob2depth(const float* prob_volume, int B, int D, int H, int W,
                    const float* depth_start, const float* depth_interval, int up, float* depth,
                    float* prob_map, atvs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ATVS_H_ */
