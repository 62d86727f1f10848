/*
 * xfeat_b200.h -- C-ABI of libxfeat_sm100.so: the XFeat inference hot path as sm_100a CUDA kernels.
 *
 * The reference (verlab/accelerated_features) has no FFI / plugin interface of its own: its boundary is the
 * Python surface of modules/xfeat.py (SURVEY.md section 8b).  Each entry point below replaces the ATen call
 * sequence of one reference function; the citation after "replaces:" is the reference file:line.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller (PyTorch allocates, we never free it);
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, no entry point synchronises
 *     the device, none allocates device memory except xfeat_create;
 *   - return value: 0 = ok, otherwise an XF_E_* code; xfeat_last_error() gives the message (thread local);
 *   - activations are channels-last (NHWC) fp32; the dense feature map returned to the caller is
 *     (B, H/8, W/8, 64) channels-last, the keypoint heat-map is (B, H, W), reliability is (B, H/8, W/8);
 *   - H, W below are the network resolution: multiples of 32 (xfeat.py:235-236).
 */
#ifndef XFEAT_B200_H
#define XFEAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XFEAT_ABI_VERSION 2
#if defined(__GNUC__)
#define XF_API __attribute__((visibility("default")))
#else
#define XF_API
#endif

enum {
  XF_OK = 0,
  XF_E_INVALID = 1,     /* bad argument */
  XF_E_CUDA = 2,        /* CUDA runtime error (message has the cudaError string) */
  XF_E_WORKSPACE = 3,   /* workspace too small */
  XF_E_UNSUPPORTED = 4
};

/* Per-image / per-pair counts (d_n_valid, d_n_matches) carry this value when the NMS candidate buffer of that image
 * overflowed (more than H*W/4 maxima above the threshold: equal-valued plateaus pass the reference's `x == local_max` test,
 * xfeat.py:252, so there is no hard bound): nothing is returned for the image instead of an arbitrary subset. */
#define XF_N_OVERFLOW (-1)

/* pixel formats accepted by xfeat_preprocess */
enum { XF_DTYPE_F32 = 0, XF_DTYPE_U8 = 1 };

typedef struct xfeat_ctx xfeat_ctx;

XF_API int xfeat_abi_version(void);
XF_API const char* xfeat_last_error(void);
/* number of kernels of this library launched by the calling process so far (cub sort passes not included) */
XF_API unsigned long long xfeat_launch_count(void);

/* Number of floats of the packed weight blob expected by xfeat_create (layer table in csrc/layers.h;
 * accelerated_features_b200/weights.py produces it: BatchNorm folded, [tap][cin][cout] order). */
XF_API size_t xfeat_packed_weight_floats(void);

/* replaces: XFeat.__init__ / XFeatModel() + load_state_dict (xfeat.py:23-35, model.py:33-111).
 * `packed_host` is a HOST pointer to xfeat_packed_weight_floats() floats. One ctx per device. */
XF_API int xfeat_create(xfeat_ctx** out, int device, const float* packed_host, size_t n_floats);
XF_API void xfeat_destroy(xfeat_ctx* ctx);

/* ---------------------------------------------------------------------------------------------------------
 * Stage entry points (each is also what the per-kernel parity tests call with oracle tensors)
 * ------------------------------------------------------------------------------------------------------- */

/* replaces: F.interpolate(scale_factor=s, bilinear, align_corners=False) in extract_dualscale (xfeat.py:380-381)
 * (and parse_input's "/255" when div255 != 0).  Input addressed with element strides like xfeat_preprocess;
 * output NCHW fp32 (B,C,Ho,Wo) contiguous; source coordinate = (dst+0.5)*scale - 0.5 (clamped at 0), the caller
 * passes scale = float(1/scale_factor) (ATen area_pixel_compute_scale with a given scale factor). */
XF_API int xfeat_resize_bilinear(const void* d_in, int dtype, int B, int C, int Hi, int Wi, int64_t stride_b,
                                 int64_t stride_c, int64_t stride_h, int64_t stride_w, int div255, float* d_out, int Ho,
                                 int Wo, float scale_h, float scale_w, void* stream);

/* replaces: preprocess_tensor's .float() + F.interpolate(size=(H,W), bilinear) (xfeat.py:233-239) and
 * XFeatModel.forward's channel mean + InstanceNorm2d(1) (model.py:135-136).
 * Input: B images, C channels, Hi x Wi pixels, element strides (in elements) for batch/channel/row/col so that
 * both NCHW tensors and HWC numpy images are read in place.  div255 != 0 applies parse_input's "/255"
 * (xfeat.py:400-401).  Output d_xn: (B, H, W) fp32 normalised gray.  d_stats: B*2 doubles scratch. */
XF_API int xfeat_preprocess(const void* d_img, int dtype, int B, int C, int Hi, int Wi,
                     int64_t stride_b, int64_t stride_c, int64_t stride_h, int64_t stride_w, int div255,
                     int H, int W, float* d_xn, double* d_stats, void* stream);

/* xfeat_preprocess with explicit source-coordinate scales (src = (dst + 0.5) * scale - 0.5): F.interpolate(scale_factor = s) uses
 * scale = float(1 / s) whatever floor(Hi * s) is (xfeat.py:380-381), F.interpolate(size = ...) uses in / out (xfeat.py:239).  With
 * it extract_dualscale's resize (3 channels written and read back) folds into the gray conversion whenever the scaled size is
 * already a multiple of 32 (then preprocess_tensor's own resize is the identity): per-channel interpolation in ATen's operation
 * order, channel sum, division -- bit-identical to the two-step form. */
XF_API int xfeat_preprocess_scaled(const void* d_img, int dtype, int B, int C, int Hi, int Wi,
                            int64_t stride_b, int64_t stride_c, int64_t stride_h, int64_t stride_w, int div255,
                            int H, int W, float scale_h, float scale_w, float* d_xn, double* d_stats, void* stream);

/* Implementation switch of the conv layers inside xfeat_net (process-wide): 0 = fp32 CUDA-core kernels everywhere,
 * 1 = tcgen05 tensor-core kernels (split-fp16 operands, fp32 accumulation in TMEM), 2 = as 1 plus halo-patch operand
 * reuse for the 3x3 stride-1 layers.  xfeat_set_halo_desc_mode is a bring-up knob of mode 2 (1 = PTX base_offset rule). */
XF_API void xfeat_set_halo_desc_mode(int mode);
XF_API void xfeat_set_conv_impl(int impl);
XF_API int xfeat_get_conv_impl(void);
/* block1.2 -> block1.3 + skip1 of conv impl 2 (process-wide): 1 (default) = one fused tcgen05 kernel that keeps the
 * half-resolution activation in shared memory, 0 = the two-kernel path.  XFEAT_BLOCK1_UNFUSED=1 in the environment forces 0;
 * xfeat_get_block1_fused reports the path in effect.  Both paths give bit-identical results. */
XF_API void xfeat_set_block1_fused(int on);
XF_API int xfeat_get_block1_fused(void);
XF_API size_t xfeat_net_workspace_bytes(int B, int H, int W);
/* replaces: XFeatModel.forward (model.py:123-154) minus the normalisation (done by xfeat_preprocess), plus
 * get_kpts_heatmap (xfeat.py:242-247) fused after keypoint_head.
 *   d_xn (B,H,W) -> d_feats (B,H/8,W/8,64) NHWC, d_heat (B,H,W), d_reliability (B,H/8,W/8),
 *   d_kpt_logits (B,H/8,W/8,65) optional (NULL to skip; tests only). */
XF_API int xfeat_net(xfeat_ctx* ctx, const float* d_xn, int B, int H, int W, float* d_feats, float* d_heat,
              float* d_reliability, float* d_kpt_logits, void* d_ws, size_t ws_bytes, void* stream);

XF_API size_t xfeat_sparse_workspace_bytes(int B, int H, int W, int top_k);
/* replaces: F.normalize(M1,dim=1), NMS, nearest*bilinear scores, argsort/top-k, bicubic descriptor sampling,
 * F.normalize(dim=-1), keypoint rescale and the `scores > 0` filter (xfeat.py:70-103).
 * Outputs (fixed capacity top_k per image, sorted by score descending, ties by raster index ascending):
 *   d_kpts (B,top_k,2) f32 = (x*rw, y*rh); d_scores (B,top_k); d_desc (B,top_k,64); d_n_valid (B) int32 = number
 *   of leading entries with score > 0, or XF_N_OVERFLOW when more than H*W/4 candidates with a positive score were found
 *   (all outputs of that image are then zero-filled); d_n_cand (B) int32 = number of NMS maxima above threshold (before the
 *   score filter; for parity checks, may be NULL); d_kpts_int (B,top_k,2) int32 optional. Entries past n_valid
 *   are zero-filled. */
XF_API int xfeat_detect_sparse(xfeat_ctx* ctx, const float* d_feats, const float* d_heat, const float* d_reliability,
                        int B, int H, int W, int top_k, float threshold, float rw, float rh,
                        float* d_kpts, float* d_scores, float* d_desc, int32_t* d_n_valid, int32_t* d_n_cand,
                        int32_t* d_kpts_int, void* d_ws, size_t ws_bytes, void* stream);

/* xfeat_detect_sparse that ALSO writes the matcher's operand rows: d_desc_split (B, split_rows, 128) fp16 = [hi(64) | lo(64)] of
 * descriptor * 2^13 (x = hi + lo; XF_DESC_SPLIT_SCALE_LOG2), rows past n_valid zero; split_rows a multiple of 512, >= top_k.
 * xfeat_mnn_match_presplit consumes them, which removes the max-reduction and split passes of xfeat_mnn_match from the sparse
 * path.  d_desc_split == NULL: identical to xfeat_detect_sparse.  d_desc may be NULL when d_desc_split is given (a caller that only
 * matches does not need the fp32 descriptors: 134 MB of writes less per 128 x 4096 keypoints). */
#define XF_DESC_SPLIT_SCALE_LOG2 13
XF_API int xfeat_detect_sparse_split(xfeat_ctx* ctx, const float* d_feats, const float* d_heat, const float* d_reliability,
                              int B, int H, int W, int top_k, float threshold, float rw, float rh, float* d_kpts,
                              float* d_scores, float* d_desc, int32_t* d_n_valid, int32_t* d_n_cand, int32_t* d_kpts_int,
                              void* d_desc_split, int split_rows, void* d_ws, size_t ws_bytes, void* stream);

XF_API size_t xfeat_dense_workspace_bytes(int B, int H, int W, int top_k);
/* replaces: extractDense's topk over the reliability map + gathers + rescale (xfeat.py:366-375) and
 * extract_dualscale's "/s" (xfeat.py:388).  k = min(top_k, (H/8)*(W/8)).
 * Writes k rows per image at row offset `out_offset` of outputs with `out_rows` rows per image:
 *   d_kpts (B,out_rows,2) = (x*8*rw/div_scale, y*8*rh/div_scale); d_desc (B,out_rows,64) un-normalised;
 *   d_scales (B,out_rows) = scale_value (xfeat.py:389-391; may be NULL); order = reliability descending, ties by cell
 *   index ascending. d_topk_idx (B,k) int32 optional. */
XF_API int xfeat_detect_dense(xfeat_ctx* ctx, const float* d_feats, const float* d_reliability, int B, int H, int W,
                       int top_k, float rw, float rh, float div_scale, float scale_value, int out_rows, int out_offset,
                       float* d_kpts, float* d_desc, float* d_scales, int32_t* d_topk_idx, void* d_ws, size_t ws_bytes,
                       void* stream);

/* Implementation switch of xfeat_mnn_match (process-wide): 0 = fp32 CUDA-core kernel; 1 = tcgen05 tensor-core kernel
 * (split-fp16 operands, fp32 accumulation in TMEM, one three-term GEMM per direction; default); 2 = tcgen05, single GEMM with the
 * column arg-max reduced in the epilogue; 3 = implementation 1 on CTA pairs (tcgen05 cta_group::2); 4 = filter +
 * exact re-score: one fp16 pass per direction tracking top-1 / top-2, then implementation 1's kernel only on the rows whose
 * gap is within the rounding bound of the dropped split terms.  All honour the same tie rule; 1-4 return identical results.
 * Values outside 0..4 are clamped. */
XF_API void xfeat_set_mnn_impl(int impl);
XF_API int xfeat_get_mnn_impl(void);
XF_API size_t xfeat_mnn_workspace_bytes(int batch, int n1_max, int n2_max);
/* replaces: XFeat.match (xfeat.py:327-348) and XFeat.batch_match (xfeat.py:265-290).
 * Batched mutual-nearest-neighbour on dot products: for pair b, rows d_f1 + b*stride1 (n1[b] x 64) against
 * d_f2 + b*stride2 (n2[b] x 64); strides in floats.  d_n1 / d_n2: device int32 per-pair counts (NULL = n1_max /
 * n2_max for every pair).  argmax ties resolve to the lowest index, as torch.max / argmax on CPU.
 * min_cossim <= 0 disables the threshold (reference semantics).
 * Outputs per pair at capacity n1_max: d_idx0, d_idx1 (batch, n1_max) int64 (idx0 ascending), d_n_matches (batch);
 * a negative d_n1 / d_n2 entry (XF_N_OVERFLOW from xfeat_detect_sparse) gives d_n_matches = XF_N_OVERFLOW for that pair.
 * Never materialises the similarity matrix. */
XF_API int xfeat_mnn_match(const float* d_f1, const int32_t* d_n1, int n1_max, int64_t stride1,
                    const float* d_f2, const int32_t* d_n2, int n2_max, int64_t stride2,
                    int batch, float min_cossim, int64_t* d_idx0, int64_t* d_idx1, int32_t* d_n_matches,
                    void* d_ws, size_t ws_bytes, void* stream);
/* xfeat_mnn_match with a caller-supplied bound: abs_bound > 0 promises max |d_f1|, max |d_f2| <= abs_bound (1.0 for the
 * unit-norm descriptors xfeat_detect_sparse writes), so the tensor-core implementations take their power-of-two operand
 * scale from it instead of running a max-reduction over both descriptor sets first.  abs_bound <= 0: identical to
 * xfeat_mnn_match.  The bound only selects the scale; results do not depend on it beyond accumulation-noise ties. */
XF_API int xfeat_mnn_match_bounded(const float* d_f1, const int32_t* d_n1, int n1_max, int64_t stride1,
                            const float* d_f2, const int32_t* d_n2, int n2_max, int64_t stride2,
                            int batch, float min_cossim, float abs_bound, int64_t* d_idx0, int64_t* d_idx1,
                            int32_t* d_n_matches, void* d_ws, size_t ws_bytes, void* stream);

/* xfeat_mnn_match on operands the producer already split (xfeat_detect_sparse_split): d_f1s / d_f2s (batch, n_pad, 128) fp16 rows
 * [hi(64) | lo(64)] of descriptor * 2^scale_log2.  Same outputs and tie rule as xfeat_mnn_match; implementations 1 and 3 only
 * (XF_E_UNSUPPORTED otherwise). */
XF_API size_t xfeat_mnn_presplit_workspace_bytes(int batch, int n1_max, int n2_max);
XF_API int xfeat_mnn_match_presplit(const void* d_f1s, const int32_t* d_n1, int n1_max, const void* d_f2s, const int32_t* d_n2,
                             int n2_max, int n_pad, int batch, int scale_log2, float min_cossim, int64_t* d_idx0,
                             int64_t* d_idx1, int32_t* d_n_matches, void* d_ws, size_t ws_bytes, void* stream);

/* Gather matched keypoints: out0[b][m] = kpts0[b][idx0[b][m]], out1[b][m] = kpts1[b][idx1[b][m]] for m < n_matches[b]
 * (replaces the fancy-indexing at xfeat.py:186). kpts are (batch, n_max, 2) f32. */
XF_API int xfeat_gather_matches(const float* d_kpts0, const float* d_kpts1, int n1_max, int n2_max,
                         const int64_t* d_idx0, const int64_t* d_idx1, const int32_t* d_n_matches, int batch,
                         float* d_out0, float* d_out1, void* stream);

XF_API size_t xfeat_refine_workspace_bytes(int batch, int n_max);
/* replaces: XFeat.refine_matches + fine_matcher + subpix_softmax2d (xfeat.py:292-325, model.py:97-111), for all
 * pairs of the batch at once.  Inputs: un-normalised coarse descriptors d_desc0 (batch,n_max,64) / d_desc1 (batch,n1_max,64),
 * keypoints d_kpts0 (batch,n_max,2) / d_kpts1 (batch,n1_max,2), d_scales0 (batch,n_max), coarse matches d_idx0/d_idx1
 * (batch,n_max) + d_n_matches (the two image sets may yield different numbers of coarse features, as reference batch_match
 * allows).  Output d_matches (batch,n_max,4) = (x0+dx*s, y0+dy*s, x1, y1) for rows with conf > fine_conf, order preserved;
 * d_n_refined (batch). */
XF_API int xfeat_refine(xfeat_ctx* ctx, const float* d_desc0, const float* d_desc1, const float* d_kpts0,
                 const float* d_kpts1, const float* d_scales0, const int64_t* d_idx0, const int64_t* d_idx1,
                 const int32_t* d_n_matches, int batch, int n_max, int n1_max, float fine_conf, float* d_matches,
                 int32_t* d_n_refined, void* d_ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stand-alone forms of the reference's helper methods (the same arithmetic runs fused inside the stage entry points)
 * ------------------------------------------------------------------------------------------------------- */

/* replaces: XFeat.get_kpts_heatmap (xfeat.py:242-247).  d_logits (B,65,Hc,Wc) NCHW fp32 -> d_heat (B,1,8*Hc,8*Wc):
 * softmax(logits * softmax_temp) over the 65 channels, dustbin dropped, heat[b,8h+i,8w+j] = p[b,8i+j,h,w]. */
XF_API int xfeat_kpts_heatmap(const float* d_logits, int B, int Hc, int Wc, float softmax_temp, float* d_heat, void* stream);

/* replaces: XFeat.NMS (xfeat.py:249-263): pos = (x == MaxPool2d(kernel_size, stride 1, pad kernel_size/2)(x)) & (x > threshold),
 * positions (x, y) int64 in raster order.  Two calls, as the reference's own nonzero() needs the count on the host:
 * xfeat_nms_count fills d_counts (B) int32; the caller sizes d_pos (B, pos_cap, 2) (zero-initialised = the reference's
 * padding, pos_cap = max count) and xfeat_nms_write fills it.  d_ws: xfeat_nms_workspace_bytes, kept between the calls. */
XF_API size_t xfeat_nms_workspace_bytes(int B, int H, int W);
XF_API int xfeat_nms_count(const float* d_heat, int B, int H, int W, int kernel_size, float threshold, int32_t* d_counts,
                           void* d_ws, size_t ws_bytes, void* stream);
XF_API int xfeat_nms_write(const float* d_heat, int B, int H, int W, int kernel_size, float threshold, int64_t* d_pos,
                           int pos_cap, void* d_ws, size_t ws_bytes, void* stream);

/* replaces: InterpolateSparse2d.forward (interpolator.py:17-33): grid = 2*pos/(W-1,H-1) - 1, F.grid_sample(align_corners=False,
 * zeros padding); mode 0 = nearest, 1 = bilinear, 2 = bicubic.  d_x (B,C,Hm,Wm) NCHW fp32, d_pos (B,N,2) fp32 (x,y) in the
 * H x W frame, d_out (B,N,C). */
XF_API int xfeat_interpolate_sparse(const float* d_x, const float* d_pos, int B, int C, int Hm, int Wm, int N, int H, int W,
                                    int mode, float* d_out, void* stream);

/* replaces: XFeat.subpix_softmax2d (xfeat.py:292-304) for 8x8 maps: d_maps (n,64) -> d_out (n,2) = E[(x-4, y-4)] under
 * softmax(temp * map). */
XF_API int xfeat_subpix_softmax2d(const float* d_maps, int64_t n, float temp, float* d_out, void* stream);

/* replaces: XFeatModel.fine_matcher (model.py:97-111; Linear + BatchNorm1d(affine=False) folded + ReLU x4, Linear):
 * d_x (n,128) -> d_out (n,64) logits. */
XF_API size_t xfeat_fine_matcher_workspace_bytes(int n);
XF_API int xfeat_fine_matcher(xfeat_ctx* ctx, const float* d_x, int n, float* d_out, void* d_ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Geometric verification right after the path (SURVEY 8f-3)
 * ------------------------------------------------------------------------------------------------------- */

/* replaces: cv2.findHomography(pts1, pts2, cv2.USAC_MAGSAC, thr, maxIters, confidence) as called on the matches by
 * realtime_demo.py:225 and the notebooks (the estimator itself lives in un-vendored OpenCV).  For every pair b:
 * d_pts0 / d_pts1 (batch, n_max, 2) matched coordinates (e.g. the outputs of xfeat_gather_matches), d_n (batch) counts (NULL:
 * n_max each).  `iters` minimal 4-point hypotheses per pair, scored on all correspondences (MSAC, forward transfer error in
 * pixels of image 1 against thr_px), best one re-fitted twice by least squares on its inliers.  Outputs: d_H (batch, 9)
 * row-major with H[8] = 1, d_inliers (batch, n_max) 0/1, d_n_inliers (batch).  Fewer than 4 matches: identity, no inliers.
 * n_max <= 8192.  Deterministic for a given seed. */
XF_API size_t xfeat_ransac_workspace_bytes(int batch, int iters);
XF_API int xfeat_ransac_homography(const float* d_pts0, const float* d_pts1, const int32_t* d_n, int n_max, int batch,
                                   float thr_px, int iters, uint32_t seed, float* d_H, uint8_t* d_inliers,
                                   int32_t* d_n_inliers, void* d_ws, size_t ws_bytes, void* stream);

/* replaces: the relative-pose RANSAC the 1500-pair benchmarks run on the matches (poselib.estimate_relative_pose,
 * modules/eval/megadepth1500.py:98-113): essential matrix from NORMALISED image coordinates d_x0 / d_x1 (batch, n_max, 2)
 * (K^-1 applied by the caller), 8-point hypotheses projected onto the essential manifold, Sampson distance against `thr` (in
 * normalised units: pixels / focal length), MSAC scoring, two least-squares re-fits.  Outputs d_E (batch, 9) row-major with
 * x1^T E x0 = 0, d_inliers, d_n_inliers.  Fewer than 8 matches: zero matrix.  (The 8-point solver is degenerate for planar
 * scenes, unlike poselib's 5-point solver.)  Workspace: xfeat_ransac_workspace_bytes. */
XF_API int xfeat_ransac_essential(const float* d_x0, const float* d_x1, const int32_t* d_n, int n_max, int batch, float thr,
                                  int iters, uint32_t seed, float* d_E, uint8_t* d_inliers, int32_t* d_n_inliers, void* d_ws,
                                  size_t ws_bytes, void* stream);

/* Test hook: run one folded conv layer of the packed table (index into csrc/layers.h) through the generic
 * kernels. in (B,Hi,Wi,Cin) NHWC -> out (B,Ho,Wo,Cout). */
XF_API int xfeat_debug_conv_layer(xfeat_ctx* ctx, int layer, const float* d_in, int B, int Hi, int Wi, float* d_out,
                           void* stream);

/* Test hook: one 64->64 stride-1 layer through the tensor-core kernel, fp32 NHWC in/out; d_scratch >= B*H*W*256 bytes. */
XF_API int xfeat_debug_conv_layer_tc(xfeat_ctx* ctx, int layer, const float* d_in, int B, int H, int W, float* d_out,
                                     void* d_scratch, size_t scratch_bytes, void* stream);

/* Test hook: block1.2 -> block1.3 + skip1 on the tensor cores (the path xfeat_set_block1_fused selects).  d_a2
 * (B,H/2,W/2,8) fp32 NHWC block1.1 output, d_xn (B,H,W) -> d_x1s (B,H/4,W/4,24) = block1(x) + skip1(x); H, W multiples of 4;
 * d_scratch >= B*(H/2)*(W/2)*64 bytes. */
XF_API int xfeat_debug_block1_tail(xfeat_ctx* ctx, const float* d_a2, const float* d_xn, int B, int H, int W, float* d_x1s,
                                   void* d_scratch, size_t scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XFEAT_B200_H */
