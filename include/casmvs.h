/*
 * casmvs.h — C ABI of libcasmvs.so, the B200 (sm_100a) cascade-MVS depth engine.
 *
 * The reference (kwea123/CasMVSNet_pl) has NO FFI layer: its boundary for the
 * hot path is the Python surface models/mvsnet.py + models/modules.py
 * (SURVEY.md §8b).  This header is the C boundary a binding for that surface
 * needs; each entry cites the reference code it replaces (paths relative to
 * the reference root).  The Python binding that mirrors the reference API on
 * top of it lives in casmvsnet_pl_b200/models/ and is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; casmvs_last_error()
 *    returns a thread-local description.  No exceptions cross the boundary.
 *  - all tensor arguments are raw DEVICE pointers owned by the caller (e.g.
 *    torch.Tensor.data_ptr()); the library never allocates or frees
 *    user-visible memory.  Scratch memory is passed in as workspace.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *    the call returns without synchronising (CUDA-graph capturable).
 *  - fp32 everywhere (the reference declares AMP unsupported, opt.py:69-70);
 *    depth_index is int64 like torch's .long().
 *  - there is no CPU fallback: casmvs_device_check() fails on anything below
 *    compute capability 10.0.
 *
 * Memory layouts (enum casmvs_layout)
 *   CASMVS_NCHW : channels-first, the reference's public layout
 *                 features (B,V,C,h,w), volumes (B,C,D,h,w)
 *   CASMVS_NHWC : channels-last, the engine's internal layout
 *                 features (B,V,h,w,C), volumes (B,D,h,w,C)
 */
#ifndef CASMVS_H_
#define CASMVS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CASMVS_VERSION 100  /* 0.1.0 */

enum casmvs_layout { CASMVS_NCHW = 0, CASMVS_NHWC = 1 };
/* OR-ed into casmvs_warp_cost_fwd's cost_layout: store the cost volume rounded to
 * TF32 (round-to-nearest) because the consumer is the tcgen05 kind::tf32 conv, which
 * would otherwise truncate the operand (biased). */
#define CASMVS_ROUND_TF32 256

/* precision of the 3D-conv contraction (K2) */
enum casmvs_precision {
  CASMVS_FP32 = 0,  /* CUDA-core fp32 FMA (bit-faithful products)            */
  CASMVS_TF32 = 1   /* tcgen05 kind::tf32, fp32 accumulate in TMEM           */
};

/* OR-ed into casmvs_conv3d_fwd's precision: store the output unrounded even in the TF32
 * mode (by default activations are stored TF32-rounded there because the next tensor-core
 * layer would otherwise truncate them; the last layer before a non-tensor consumer should
 * keep the fp32 accumulator). */
#define CASMVS_KEEP_FP32_OUT 256

enum casmvs_conv_kind {
  CASMVS_CONV = 0,           /* Conv3d(k=3, pad=1, stride 1|2)   modules.py:26      */
  CASMVS_CONV_TRANSPOSE = 1, /* ConvTranspose3d(k=3,s=2,p=1,op=1) mvsnet.py:75,80,85 */
  /* 1x3x3 kernel, stride 1, pad (0,1,1): the 3x3 Conv2d layers of FeatureNet
   * (ConvBnReLU modules.py:8-18, smooth0/1 mvsnet.py:30-31) run as ONE convolution over
   * the (views, H, W) volume of a batch.  Packed weights keep the [27][Cin][Cout] layout
   * with zero kd = 0 and kd = 2 planes, so every K2 kernel computes it correctly and the
   * tensor-core kernels skip the two empty planes. */
  CASMVS_CONV_PLANAR = 2
};

/* ---- library / device ------------------------------------------------- */
int casmvs_version(void);
const char* casmvs_last_error(void);
/* 0 iff `device` exists and has compute capability >= 10.0 (no fallback). */
int casmvs_device_check(int device);
/* number of kernels this library has launched since load (bench evidence). */
uint64_t casmvs_launch_count(void);
/* number of CASMVS_TF32 layers that no tcgen05 kernel covered and that therefore ran on the
 * CUDA-core kernel (same results up to TF32 rounding, several times slower).  0 for the
 * reference architecture at every BASELINE configuration; bench.py and the full-size tests
 * assert that. */
uint64_t casmvs_fallback_count(void);

/* ---- K1: fused homography warp + bilinear sample + cost reduction ------
 * Replaces homo_warp (models/modules.py:52-92) called V-1 times plus the
 * variance (models/mvsnet.py:137-141,147-156,166-168) or group-wise
 * correlation (:143-144,158-162,170-172) accumulation.  The warped
 * (B,V-1,C,D,h,w) volumes are never materialised.
 *   feats        (B,V,C,h,w) [NCHW] or (B,V,h,w,C) [NHWC]; view 0 = reference
 *   proj         (B,V-1,3,4) row-major  src_proj @ ref_proj^-1
 *   depth_values (B,D,h,w)
 *   cost         num_groups==1: C channels  (B,C,D,h,w)|(B,D,h,w,C)
 *                num_groups >1: G channels  (B,G,D,h,w)|(B,D,h,w,G)
 * Workspace: casmvs_warp_cost_workspace_bytes() (only needed when feats are
 * NCHW: they are re-laid-out once to NHWC).  C % 8 == 0, C % G == 0.
 */
size_t casmvs_warp_cost_workspace_bytes(int feat_layout, int B, int V, int C, int h, int w);
int casmvs_warp_cost_fwd(const float* feats, int feat_layout, const float* proj,
                         const float* depth_values, float* cost, int cost_layout,
                         int B, int V, int C, int D, int h, int w, int num_groups,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Stand-alone homo_warp (models/modules.py:52-92): materialises the warped
 * volume for API completeness.  src_feat (B,C,h,w)|(B,h,w,C), proj (B,3,4),
 * depth_values (B,D,h,w) -> warped (B,C,D,h,w)|(B,D,h,w,C).               */
int casmvs_homo_warp_fwd(const float* src_feat, int feat_layout, const float* proj,
                         const float* depth_values, float* warped, int out_layout,
                         int B, int C, int D, int h, int w, void* stream);

/* ---- K2: 3x3x3 convolution with fused norm-act epilogue ----------------
 * Replaces ConvBnReLU3D (models/modules.py:21-31), the ConvTranspose3d +
 * norm_act pairs and the skip additions of CostRegNet.forward
 * (models/mvsnet.py:60-104) and its `prob` head (:89,103).
 *   y = act( conv(x, w) * scale[c] + shift[c] ) + skip
 *   act(v) = v >= 0 ? v : slope * v   (slope = 1 -> identity, used by `prob`)
 * Volumes are channels-last (B,D,h,w,C).  Weights are pre-packed with
 * casmvs_pack_conv3d_weights (tap-major [27][Cin][Cout]).
 * For kind == CASMVS_CONV: stride in {1,2}, out dims = (in-1)/stride+1.
 * For kind == CASMVS_CONV_TRANSPOSE: out dims = 2*in.
 * For kind == CASMVS_CONV_PLANAR: stride 1, out dims = in dims.
 */
size_t casmvs_packed_conv3d_weight_floats(int Cin, int Cout);
/* w_torch: Conv3d layout (Cout,Cin,3,3,3), ConvTranspose3d layout (Cin,Cout,3,3,3) or, for
 * CASMVS_CONV_PLANAR, Conv2d layout (Cout,Cin,3,3) */
int casmvs_pack_conv3d_weights(const float* w_torch, int kind, int Cin, int Cout,
                               float* w_packed, void* stream);
/* The tensor-core kernels keep a per-process cache of operand images keyed by the w_packed
 * pointer (thread-safe).  An image lives as long as the packed buffer it was built from:
 *   casmvs_release_weight_images(p, bytes) drops the images whose key lies in [p, p+bytes);
 *     call it when a packed buffer is (re)created at an address, rewritten in place or freed
 *     (frees device memory => synchronises with kernels still reading those images);
 *   casmvs_invalidate_weight_cache() drops everything;
 *   casmvs_weight_cache_generation() increases whenever at least one image was dropped: a
 *     captured CUDA graph embeds image pointers and must be re-captured when it changes. */
int casmvs_release_weight_images(const void* w_packed, size_t bytes);
int casmvs_invalidate_weight_cache(void);
uint64_t casmvs_weight_cache_generation(void);
/* number of cached images keyed inside [w_packed, w_packed + bytes): a captured graph records
 * it per packed buffer it depends on and re-checks it before every replay (a release anywhere
 * else -- another model, a dead model's recycled address -- does not invalidate the graph). */
int casmvs_weight_image_count(const void* w_packed, size_t bytes);
/* Synchronises the device and marks every cached image as built.  Call it between the warm-up
 * forward and a CUDA-graph capture: during a capture the cache cannot query or wait on the
 * builders' events (such calls invalidate the capture), so it must already know. */
int casmvs_settle_weight_images(void);
int casmvs_conv3d_fwd(const float* x, const float* w_packed, const float* scale,
                      const float* shift, float slope, const float* skip, float* y,
                      int B, int Cin, int Cout, int D, int h, int w, /* INPUT dims */
                      int kind, int stride, int precision, void* stream);

/* Whole CostRegNet (models/mvsnet.py:91-104) in one call.  `params` is a
 * device array produced by casmvs_costreg_pack (see casmvs_costreg_param_floats).
 * x (B,D,h,w,Cin) -> logits (B,D,h,w) ; D,h,w divisible by 8.                */
size_t casmvs_costreg_param_floats(int Cin);
/* Layout of the params blob: layers 0..10 = conv0..conv6, conv7, conv9, conv11,
 * prob; each is packed weights [27][cin][cout], scale[cout], shift[cout]
 * (scale/shift = folded eval-mode ABN: alpha = gamma/sqrt(var+eps),
 * beta' = beta - mean*alpha; prob: scale = 1, shift = bias).  Offsets in floats. */
int casmvs_costreg_layer_info(int Cin, int layer, int* cin, int* cout, int* kind, int* stride,
                              size_t* w_off, size_t* scale_off, size_t* shift_off);
size_t casmvs_costreg_workspace_bytes(int B, int Cin, int D, int h, int w);
int casmvs_costreg_fwd(const float* x, const float* params, float* logits,
                       int B, int Cin, int D, int h, int w, int precision,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- K3: softmax over D + depth regression + index + confidence --------
 * Replaces F.softmax + depth_regression (models/mvsnet.py:174-177,
 * models/modules.py:95-104) and the confidence block (:179-193).
 *   logits (B,D,h,w); depth_values (B,D,h,w) or, if dv_is_vector, (D,)
 *   depth (B,h,w) f32, confidence (B,h,w) f32,
 *   index (B,h,w) int64 or NULL, prob (B,D,h,w) or NULL.
 * input_is_prob != 0 skips the softmax (logits already hold probabilities).
 * Sums over D use the main-path order of ATen's CPU sum (sequential 16-term
 * chunks, cascaded); depth_index equals the oracle's for identical p.      */
int casmvs_regress_fwd(const float* logits, const float* depth_values, int dv_is_vector,
                       int input_is_prob, float* depth, float* confidence,
                       int64_t* index, float* prob, int B, int D, int h, int w,
                       void* stream);

/* ---- K4: depth hypotheses ----------------------------------------------
 * casmvs_depth_hypotheses_fwd replaces get_depth_values
 * (models/modules.py:34-49): out[b,d] = max(cur - half_range, 1e-7) + step*d.
 * If upsample != 0 `cur` is (B,h/2,w/2) and is first upsampled x2 bilinear,
 * align_corners=True (models/mvsnet.py:231-234); else `cur` is (B,h,w).
 * step_dev (B floats, device) overrides `step`/`half_range` when non-NULL
 * (tensor-valued depth_interval): half_range = fl32(D/2)*step_dev[b].
 * casmvs_uniform_hypotheses_fwd replaces models/mvsnet.py:213-229:
 * out[b,d,:,:] = depth_min + step*d, depth_min/step scalars or device (B,).  */
int casmvs_depth_hypotheses_fwd(const float* cur, int upsample, float half_range,
                                float step, const float* step_dev, float* out,
                                int B, int D, int h, int w, void* stream);
int casmvs_uniform_hypotheses_fwd(float depth_min, float step, const float* depth_min_dev,
                                  const float* step_dev, float* out,
                                  int B, int D, int h, int w, void* stream);

/* ---- cascade-internal forms: hypotheses as a ladder, never materialised -----------------
 * Inside the cascade every pixel's hypotheses are first + step*d (get_depth_values,
 * models/modules.py:44-48; initial planes, models/mvsnet.py:215-229).  These entries take the
 * ladder instead of the (B,D,h,w) tensor and generate it in the kernel with the same two
 * roundings, so K4's D*h*w floats are neither written nor read back by K1 and K3 (bit-identical
 * results).  first: `first_map` (B,h,w) per pixel, else `first_b` (B) per batch item, else the
 * scalar `first`; step: `step_b` (B) else the scalar `step`.
 * casmvs_depth_first_fwd writes only the first rung (B,h,w) of casmvs_depth_hypotheses_fwd.
 * casmvs_warp_cost_ladder_fwd: channels-last features and cost volume; shapes of the staged
 * kernel only (V-1 in {1,2}, C in {8,16,32}, num_groups 1 or 8), error otherwise. */
int casmvs_depth_first_fwd(const float* cur, int upsample, float half_range, float step,
                           const float* step_dev, float* out, int B, int D, int h, int w,
                           void* stream);
int casmvs_warp_cost_ladder_fwd(const float* feats, const float* proj, const float* first_map,
                                const float* first_b, float first, const float* step_b, float step,
                                float* cost, int round_tf32, int B, int V, int C, int D, int h, int w,
                                int num_groups, void* stream);
int casmvs_regress_ladder_fwd(const float* logits, const float* first_map, const float* first_b,
                              float first, const float* step_b, float step, float* depth,
                              float* confidence, int64_t* index, int B, int D, int h, int w,
                              void* stream);

/* ---- FeatureNet top-down path, fused (adjacent to the hot path; SURVEY.md §8f-2) ----
 * One pyramid level of models/mvsnet.py:36-52:
 *   feat = upsample_x2_bilinear(prev, align_corners=True) + conv1x1(c, lat_w) + lat_b   (32 ch)
 *   out  = conv3x3(feat, smooth_w, pad 1) + smooth_b
 * prev (N,h/2,w/2,32), c (N,h,w,CLAT), out (N,h,w,COUT), feat_out (N,h,w,32) or NULL; all
 * channels-last.  lat_w (32,CLAT[,1,1]) and smooth_w (COUT,32,3,3) in torch layout. */
int casmvs_fpn_level_fwd(const float* prev, const float* c, const float* lat_w,
                         const float* lat_b, const float* smooth_w, const float* smooth_b,
                         float* feat_out, float* out, int N, int h, int w, int CLAT, int COUT,
                         void* stream);

/* The same level split in two for the tensor-core path: this call produces
 *   feat = upsample_x2_bilinear(prev, align_corners=True) + conv1x1(c, lat_w) + lat_b
 * (N,h,w,32), optionally TF32-rounded, and the 3x3 smooth runs as a CASMVS_CONV_PLANAR
 * casmvs_conv3d_fwd on tcgen05.  prev == NULL: feat = conv1x1(c) + lat_b (the `toplayer`,
 * mvsnet.py:27,41).  lat_w (32,CLAT[,1,1]) torch layout; CLAT % 4 == 0. */
int casmvs_fpn_merge_fwd(const float* prev, const float* c, const float* lat_w,
                         const float* lat_b, float* feat, int N, int h, int w, int CLAT,
                         int round_tf32, void* stream);

/* First FeatureNet block (ConvBnReLU(3, 8, 3, 1, 1), mvsnet.py:13 + modules.py:8-18) with the
 * eval-mode ABN folded: y = LeakyReLU(conv3x3(x, w, pad 1) + bias).  x (N,3,H,W) planar fp32
 * (the image batch as the data loader hands it over, no re-layout), w (8,3,3,3) torch
 * layout already multiplied by the ABN scale, y (N,H,W,8) channels-last. */
int casmvs_conv2d_rgb8_fwd(const float* x, const float* w, const float* bias, float slope,
                           float* y, int N, int H, int W, int round_tf32, void* stream);

/* The 5x5 stride-2 blocks of FeatureNet (ConvBnReLU(8,16,5,2,2) / (16,32,5,2,2), mvsnet.py:16,20
 * + modules.py:8-18) with the eval-mode ABN folded, on tcgen05 (TF32 operands):
 *   y = LeakyReLU(conv5x5_s2_p2(x, w) + shift)
 * x (N,H,W,Cin) channels-last, w (Cout,Cin,5,5) torch layout already multiplied by the ABN
 * scale, y (N,(H-1)/2+1,(W-1)/2+1,Cout) channels-last, optionally stored TF32-rounded.  The
 * operand image built from `w` is cached by pointer (casmvs_invalidate_weight_cache). */
int casmvs_conv2d_5x5s2_fwd(const float* x, const float* w, const float* shift, float slope,
                            float* y, int N, int Cin, int Cout, int H, int W, int round_tf32,
                            void* stream);

/* The same blocks in the fp32 precision mode: CUDA-core FMA, bit-faithful products, output
 * unrounded.  Same layouts; w is the plain (Cout,Cin,5,5) torch tensor (nothing is cached). */
int casmvs_conv2d_5x5s2_fp32_fwd(const float* x, const float* w, const float* shift, float slope,
                                 float* y, int N, int Cin, int Cout, int H, int W, void* stream);

/* In-place x[...,c] = LeakyReLU(x[...,c] + bias[c]) on a channels-last tensor (C % 4 == 0):
 * the epilogue of a folded conv + eval-mode ABN block (models/modules.py:8-18). */
int casmvs_bias_lrelu_nhwc(float* x, const float* bias, float slope, size_t numel, int C,
                           void* stream);
/* Same, optionally storing the result TF32-rounded (round to nearest) for a tensor-core
 * consumer that would otherwise truncate it. */
int casmvs_bias_act_nhwc(float* x, const float* bias, float slope, size_t numel, int C,
                         int round_tf32, void* stream);

/* ---- backward of the hot path (SURVEY.md 8 f-1; reference train.py:99-127) -----------------
 * casmvs_warp_cost_bwd: gradient of casmvs_warp_cost_fwd w.r.t. the features (the only
 * differentiable input: hypotheses are detached, models/mvsnet.py:231).  All tensors
 * channels-last: feats (B,V,h,w,C), grad_cost (B,D,h,w,Cout), grad_feats (B,V,h,w,C) which the
 * caller ZEROES first (the bilinear taps are scattered into it with atomics).
 * casmvs_conv3d_wgrad: grad_w[27][Ca][Cb] += sum_{b,o} x[b, stride*o + k - 1, a] * grad_y[b,o,b']
 * for Conv3d (x = layer input, grad_y = output gradient, Ca = Cin, Cb = Cout) and, with the
 * roles swapped (x = output gradient, grad_y = layer input, stride 2), for ConvTranspose3d;
 * caller zeroes grad_w.  Channels <= 64.  The DATA gradients are forward kernels:
 * conv s1 -> conv s1 with flipped/transposed weights, conv s2 -> CASMVS_CONV_TRANSPOSE,
 * transposed -> conv s2 (casmvs_conv3d_fwd, scale = shift = NULL, slope = 1).
 * casmvs_regress_bwd: grad_logits = softmax(logits) * (depth_values - depth) * grad_depth. */
int casmvs_warp_cost_bwd(const float* feats, const float* proj, const float* depth_values,
                         const float* grad_cost, float* grad_feats, int B, int V, int C, int D,
                         int h, int w, int num_groups, void* stream);
int casmvs_conv3d_wgrad(const float* x, const float* grad_y, float* grad_w, int B, int Ca, int Cb,
                        int Di, int hi, int wi, int Do, int ho, int wo, int stride, void* stream);
int casmvs_regress_bwd(const float* logits, const float* depth_values, int dv_is_vector,
                       const float* grad_depth, float* grad_logits, int B, int D, int h, int w,
                       void* stream);

/* ---- input pipeline (SURVEY.md 8 f-4) -------------------------------------
 * T.ToTensor() + T.Normalize(mean, std) of the reference's data sets (datasets/dtu.py:130-137)
 * for images uploaded as bytes: images (N,H,W,3) uint8 RGB -> out (N,3,H,W) float32,
 * y = ((float)x / 255 - mean[c]) / std[c] in that operation order (bit-identical to
 * torchvision).  mean3 / std3 are HOST arrays of 3 floats.  H*W % 4 == 0 when N > 1. */
int casmvs_normalize_u8_fwd(const uint8_t* images, float* out, int N, int H, int W,
                            const float* mean3, const float* std3, void* stream);

/* PIL.Image.resize(size, Image.BILINEAR) of the same data sets (datasets/dtu.py:159-162,
 * tanks.py, blendedmvs.py:162-163), bit-exact: in (N,H,W,3) uint8 RGB -> out (N,h,w,3) uint8.
 * The taps are PIL's fixed-point coefficients, built on the host (io.pil_bilinear_coeffs):
 * per output column x, xmin_x[x] and taps_x[x*kx .. x*kx+kx) int32 weights with 22 fractional
 * bits (unused trailing taps 0); the same for rows.  All four tables are DEVICE arrays.  The
 * horizontal pass runs first and is clipped to uint8, then the vertical pass; a pass whose
 * axis keeps its size is skipped and its tables are ignored (may be NULL).  Returns an error
 * when the taps of one 16x64 output tile do not fit shared memory (a 48 KB budget; the data
 * sets need at most 4 taps per axis).  in and out must not overlap. */
int casmvs_resize_u8_fwd(const uint8_t* in, int N, int H, int W, uint8_t* out, int h, int w,
                         const int* xmin_x, const int* taps_x, int kx, const int* xmin_y,
                         const int* taps_y, int ky, void* stream);

/* ---- geometric-consistency filter + refinement + back-projection (SURVEY.md 8 f-3) ------
 * One reference view of eval.py:262-318 on the device; replaces xy_ref2src / xy_src2ref /
 * check_geo_consistency (eval.py:113-182, numba + cv2.remap on the CPU).  For every reference
 * pixel and each of the S source views: project with depth_ref, sample the source depth (and
 * image) bilinearly with cv2.remap's semantics (map rounded to 1/32 px, zero outside), lift
 * back, mask = |dp| < 1 px and |dd|/d < 1 %.
 *   depth_ref (H,W); image_ref (H,W,3) or NULL; proba_ref (H/4,W/4) or NULL (= confidence_2,
 *   upsampled x4 like cv2.resize INTER_LINEAR and compared with conf_thresh);
 *   depth_src / image_src: HOST arrays of S device pointers; proj_ref2src / proj_src2ref: HOST
 *   arrays (S,3,4) = (P_src @ inv(P_ref))[:3] / (P_ref @ inv(P_src))[:3]; ref2world (4,4) device.
 * Outputs (device): depth_refined (H,W) = (depth_ref + sum of consistent reprojections)/(n+1),
 * image_refined (H,W,3) or NULL, geo_count (H,W) int32, mask_final (H,W) uint8 or NULL
 * (geo_count >= min_consistent and confidence), points (H,W,3) world coordinates of the
 * refined depth or NULL; reproj_dbg (S,H,W) / mask_dbg (S,H,W) per-view results or NULL. */
int casmvs_geo_fuse_fwd(const float* depth_ref, const float* image_ref, const float* proba_ref,
                        const float* const* depth_src, const float* const* image_src,
                        const float* proj_ref2src, const float* proj_src2ref,
                        const float* ref2world, int S, int H, int W, float conf_thresh,
                        int min_consistent, float* depth_refined, float* image_refined,
                        int* geo_count, unsigned char* mask_final, float* points,
                        float* reproj_dbg, unsigned char* mask_dbg, void* stream);

/* ---- layout helpers ------------------------------------------------------ */
/* (N,C,S) -> (N,S,C) and back, S = product of spatial dims. */
int casmvs_nchw_to_nhwc(const float* in, float* out, int N, int C, size_t S, void* stream);
int casmvs_nhwc_to_nchw(const float* in, float* out, int N, int C, size_t S, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CASMVS_H_ */
