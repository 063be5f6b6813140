/* balf_b200 -- C-ABI of the B200-native BALF inference hot path (libbalf_b200.so).
 *
 * The reference (ericzzj1989/BALF) is pure Python and has no FFI; its drop-in boundary is the
 * Python call surface listed in SURVEY.md section 8b.  The PyTorch-facing modules under
 * balf_b200/ keep that surface and forward into the entry points below, one per stage of
 * demo/demo_match.py::extract_matches.  Each declaration cites the reference code it replaces.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked "host";
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream, never
 *    allocate, never synchronise (exception: functions documented as "host-synchronous");
 *  - return 0 on success, <0 for an argument / shape error, >0 = cudaError_t; the message is
 *    available from balf_last_error() (thread-local);
 *  - scratch memory is caller-provided: query *_workspace_bytes() first;
 *  - the library fails loudly: there is no CPU fallback anywhere.
 */
#ifndef BALF_B200_H_
#define BALF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BALF_B200_ABI_VERSION 1
#define BALF_API __attribute__((visibility("default")))

BALF_API const char* balf_last_error(void);
BALF_API int balf_abi_version(void);
/* number of kernels this library has launched since load (bench.py: "gpu_launches") */
BALF_API unsigned long long balf_launch_count(void);

/* Per-kernel timing for the roofline report (bench.py): while enabled, every kernel launch of the
 * library is bracketed by two CUDA events on the launching stream.  balf_profile_report is
 * host-synchronous: it waits for the events and writes one "name launches total_ms" line per
 * kernel name into `buf` (host).  No reference counterpart (the reference has no profiler hooks,
 * SURVEY.md section 5). */
BALF_API int balf_profile_enable(int on);
BALF_API int balf_profile_report(char* buf, size_t cap, int reset);

/* ------------------------------------------------------------------------------------------
 * D3  detector architecture + weights
 *     replaces: balf/model/mlp_ma_decoder.py:246-276 (MLP_MA_DECODER.__init__),
 *               balf/model/get_model.py:88-90 (load_model)
 * `raw` is every floating-point tensor of the reference state_dict, flattened and concatenated
 * in state_dict order (SURVEY.md appendix A: 4 x 40 Down tensors, then detector_head.dense.
 * {weight,bias}, detector_head.norm.{weight,bias,running_mean,running_var}).
 * balf_detector_pack_weights() lays them out for the kernels (transposes, BatchNorm folding). */
typedef struct balf_detector_arch {
    int32_t dims[5];        /* en_embed_dims, e.g. {3,32,64,128,256}                           */
    int32_t grid_h, grid_w; /* grid_size  (cells per image side; the kernels require 8 x 8)    */
    int32_t block_h, block_w; /* block_size (pixels per block side; the kernels require 8 x 8) */
    int32_t grid_factor, block_factor, proj_factor; /* all 2                                   */
    int32_t reduction;      /* channels_reduction (squeeze-excite), 4                          */
    int32_t cell;           /* cell_size of the head (8 -> 65 logits)                          */
} balf_detector_arch;

BALF_API int balf_detector_check_arch(const balf_detector_arch* arch);
BALF_API int64_t balf_detector_raw_weight_count(const balf_detector_arch* arch);
BALF_API int64_t balf_detector_packed_weight_count(const balf_detector_arch* arch);
BALF_API int balf_detector_pack_weights(const balf_detector_arch* arch, const float* raw, float* packed, void* stream);

/* ------------------------------------------------------------------------------------------
 * D0  image -> network input
 *     replaces: demo/demo_match.py:22-29 + balf/utils/test_utils.py:16-32
 *               (/255., make_shape_even, mod_padding_symmetric(factor), HWC->CHW)
 * balf_pad_geometry (host, pure arithmetic): padded size and the offset of the image inside it
 * (also the un-pad crop origin of demo_match.py:38-43).
 * balf_preprocess_u8: img [B,H,W,C] uint8 (C = 1 or 3; C = 1 is replicated to 3 planes)
 *     -> x [B,3,Hp,Wp] fp32 = float(u8)/255.f, zeros in the padding. */
BALF_API int balf_pad_geometry(int H, int W, int factor, int* Hp, int* Wp, int* top, int* left);
BALF_API int balf_preprocess_u8(const uint8_t* img, int B, int H, int W, int C, float* x, int Hp, int Wp, int top,
                       int left, void* stream);

/* ------------------------------------------------------------------------------------------
 * D1 + D2  detector forward
 *     replaces: balf/model/mlp_ma_decoder.py:278-285 (MLP_MA_DECODER.forward: 4 x Down,
 *               :201-244) and balf/model/decoder.py:16-30 (DetectorHead.forward) with
 *               balf/utils/tensor_op.py:1-27 (pixel_shuffle) fused in.
 * x [B,dims[0],Hp,Wp] fp32 NCHW, Hp and Wp multiples of 64.
 * logits [B,cell^2+1,Hp/8,Wp/8] (may be NULL), prob [B,Hp,Wp].
 * precision: 0 = fp32 FFMA (bit-level class of the reference's fp32 path),
 *            1 = tensor cores (tcgen05) on fp16 / tf32 operands (11-bit significand), fp32 accumulate: rel <= 1e-3,
 *            2 = tensor cores in split precision ("f16x3"): every operand an fp16 hi + lo pair, every product three MMAs
 *                (hi*hi + lo*hi + hi*lo): fp32-class score maps (measured max rel 5e-6 against precision 0). */
BALF_API size_t balf_detector_workspace_bytes(const balf_detector_arch* arch, int B, int Hp, int Wp);
BALF_API int balf_detector_forward(const balf_detector_arch* arch, const float* packed, const float* x, int B, int Hp,
                          int Wp, float* logits, float* prob, void* workspace, size_t workspace_bytes,
                          int precision, void* stream);
/* development hook, no reference counterpart: key 0 = bit mask of detector stages that run on the tensor-core
 * kernels when precision >= 1 (bits 0-3: the four Down stages, bit 4: the head; default all); key 1 = images per
 * internal pass of balf_detector_forward (default 16; query the workspace size again after changing it). */
BALF_API int balf_debug_set(int key, int value);
/* development hook: `buf` = device buffer of 8192 int64 (or NULL to switch off).  While set, CTA 0 of every tensor-core
 * detector kernel records SM-clock stamps of its first tiles' phases there (scripts/tc_trace.py reads them). */
BALF_API int balf_debug_set_trace(void* buf);
/* stand-alone depth-to-space (balf/utils/tensor_op.py:1-27): in [N,C,H,W] -> out [N,C/r^2,H*r,W*r] */
BALF_API int balf_pixel_shuffle(const float* in, float* out, int N, int C, int H, int W, int r, void* stream);

/* ------------------------------------------------------------------------------------------
 * P1-P8  score map -> keypoints.  The score map is the (padded) `prob` of the detector:
 * score [B, Hs, Ws] with the image occupying rows [top, top+H) and columns [left, left+W)
 * (un-pad crop, demo_match.py:38-43, fused).  Scores must be >= 0 (softmax probabilities).
 * Output per image (capacity k): xy int32 [B,k,2] = (x, y) in crop coordinates, score fp32
 * [B,k], count int32 [B]; rows are ordered score-descending with ties broken by raster index
 * y*W+x ascending (the canonical tie rule, SURVEY.md section 8c).
 *
 * balf_windowed_nms_topk  replaces test_utils.py:34-47 (remove_borders), :50-54 (apply_nms:
 *     size x size maximum filter, plateau ties all survive), :56-95 (get_point_coordinates /
 *     find_index_higher_scores: k-th value threshold with the raster-order truncation quirks)
 *     and the caller's argsort, balf/utils/train_utils.py:446-452.  Requires H*W >= k
 *     (the reference raises IndexError otherwise).
 * balf_greedy_nms_topk    replaces test_utils.py:34-47, :97-128 (get_points_direct_from_score_map:
 *     fp32 threshold `>= thr`), :130-168 (nms_fast: greedy, (2r+1)^2 exclusion box), :170-215
 *     (sub-pixel soft-argmax over a ps x ps window, ps = 0 disables) and demo_match.py:51-57
 *     (top-k by score).  dxdy fp32 [B,k,2] (may be NULL when ps = 0) holds the sub-pixel offset
 *     to ADD to (x, y) (already includes the "- ps/2" of test_utils.py:179). */
BALF_API size_t balf_nms_workspace_bytes(int B, int H, int W, int k);
BALF_API int balf_windowed_nms_topk(const float* score, int B, int Hs, int Ws, int top, int left, int H, int W,
                           int border, int nms_size, int k, int32_t* xy, float* out_score, int32_t* count,
                           void* workspace, size_t workspace_bytes, void* stream);
BALF_API int balf_greedy_nms_topk(const float* score, int B, int Hs, int Ws, int top, int left, int H, int W,
                         int border, float thr, int radius, int k, int subpixel_ps, int32_t* xy,
                         float* out_score, float* dxdy, int32_t* count, void* workspace,
                         size_t workspace_bytes, void* stream);

/* stand-alone pieces of the above, for callers that use the reference helpers one by one:
 * balf_apply_nms_map   test_utils.py:50-54 on a dense map [B,H,W] (border = 0 reproduces apply_nms;
 *                      border > 0 fuses remove_borders first): out = s * (s == max_filter(s, size)).
 * balf_subpixel_refine test_utils.py:170-215 for n given integer points per image (xy int32 [B,n,2])
 *                      -> dxdy fp32 [B,n,2]. */
BALF_API int balf_apply_nms_map(const float* score, int B, int H, int W, int border, int nms_size, float* out,
                                void* stream);
BALF_API int balf_subpixel_refine(const float* score, int B, int Hs, int Ws, int top, int left, int H, int W,
                                  int border, const int32_t* xy, int n, int ps, float* dxdy, void* stream);

/* balf_box_nms_map  replaces balf/benchmark_test/repeatability_tools.py:227-255 (box_nms, the fourth back end of the --nms
 *     switch of balf/configs/config_hpatches.py:25-26): prob [B,H,W] -> out [B,H,W] = prob at the pixels torchvision.ops.nms
 *     keeps (size x size boxes centred on every pixel with prob >= min_prob, IoU threshold `iou`, float32 IoU arithmetic),
 *     optionally only the keep_top_k best (<= 0: all), zero elsewhere.  Equal scores resolve in raster order.
 *     Workspace: balf_nms_workspace_bytes(B, H, W, k) + 12 * B * keep_top_k (when keep_top_k > 0). */
BALF_API int balf_box_nms_map(const float* prob, int B, int H, int W, float size, float iou, float min_prob, int keep_top_k,
                              float* out, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * F1  keypoints -> descriptor patches
 *     replaces: demo/demo_match.py:62-69 (kornia laf_from_center_scale_ori with scale s_mult and angle
 *               0, then extract_patches_from_pyramid(gray / 255., lafs, PS)) -- kornia 0.7.4 is not
 *               vendored by the reference: PARITY UNPINNED (oracle/thirdparty.py restates it).
 * gray [B,H,W] uint8, kpts fp32 [B,K,2] = (x, y) in pixels, count int32 [B] (NULL: K valid rows per
 * image) -> patches fp32 [B,K,PS,PS]; rows beyond count[b] are left untouched.
 * balf_patch_pyramid_level (host): the pyramid level every keypoint samples (1 for 60 / 32). */
BALF_API int balf_patch_pyramid_level(int H, int W, float s_mult, int PS);
BALF_API size_t balf_patches_workspace_bytes(int B, int H, int W);
BALF_API int balf_extract_patches_u8(const uint8_t* gray, int B, int H, int W, const float* kpts, const int32_t* count,
                                     int K, float s_mult, int PS, float* patches, void* workspace,
                                     size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * H1  HardNet descriptor
 *     replaces: third_party/hardnet/hardnet_pytorch.py:29-72 (HardNet.forward: input_norm, 7 conv +
 *               BatchNorm(affine=False, eval) (+ ReLU), L2Norm) and the 1000-patch chunk loop of
 *               demo/demo_match.py:71-93.
 * `raw` = every floating tensor of the HardNet state_dict concatenated in state_dict order
 * (features.{0,3,6,9,12,15,19}.weight each followed by its BatchNorm running_mean, running_var).
 * patches fp32 [N,1,32,32] -> desc fp32 [N,128].
 * precision: 0 = fp32 FFMA kernels (hardnet.cu),
 *            1 = the six 3x3 layers after the first as implicit-GEMM tcgen05 tiles, TF32 operands, fp32 accumulate
 *                in TMEM (hardnet_tc.cu),
 *            2 = the same kernels with fp16 operands (same 11-bit significand as TF32, half the bytes and half the MMAs;
 *                activations are post-ReLU and saturate at 65504); the workspace size depends on the precision. */
BALF_API int64_t balf_hardnet_raw_weight_count(void);
BALF_API int64_t balf_hardnet_packed_weight_count(void);
BALF_API int balf_hardnet_pack_weights(const float* raw, float* packed, void* stream);
BALF_API size_t balf_hardnet_workspace_bytes(int n_patches, int precision);
BALF_API int balf_hardnet_forward(const float* packed, const float* patches, int n_patches, float* desc, void* workspace,
                                  size_t workspace_bytes, int precision, void* stream);

/* ------------------------------------------------------------------------------------------
 * M1  SMNN matching
 *     replaces: demo/demo_match.py:104-108 (kornia match_smnn(desc1, desc2, 0.99)) -- kornia 0.7.4 is
 *               not vendored by the reference: PARITY UNPINNED (oracle/thirdparty.py restates it).
 * d1 fp32 [n1,dim], d2 fp32 [n2,dim], dim = 128 -> ids int32 [<=n1,2] = (index in d1, index in d2)
 * ascending in the first index, dist fp32 [<=n1] = max of the two Lowe ratios, count int32 [1].
 * dm_out (may be NULL) receives the fp32 distance matrix [n1,n2] the decisions were taken on.
 * Exactly equal distances resolve to the lower index. */
BALF_API size_t balf_match_workspace_bytes(int n1, int n2);
BALF_API int balf_match_smnn(const float* d1, int n1, const float* d2, int n2, int dim, float th, int32_t* ids,
                             float* dist, int32_t* count, float* dm_out, void* workspace, size_t workspace_bytes,
                             void* stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md section 8(f): front end and multi-scale extraction (the rows next to the hot path)
 * balf_rgb_to_gray_u8       replaces demo/demo_match.py:13-19 (PIL Image.convert('L')): rgb [B,H,W,3] uint8 ->
 *                           gray [B,H,W] uint8 = (19595 R + 38470 G + 7471 B + 32768) >> 16.
 * balf_preprocess_f32       replaces balf/utils/train_utils.py:417-430 (extract_detections: make_shape_even,
 *                           mod_padding_symmetric, HWC->CHW of an already normalised float image [B,H,W,C]).
 * balf_resize_preprocess_u8 one pyramid level of the multi-scale extraction advertised by
 *                           balf/configs/config_hpatches.py:50-82 (the reference ships only the argument parser:
 *                           the semantics are defined here and restated in oracle/multiscale.py, PARITY UNPINNED):
 *                           bilinear resize of the uint8 image to Hs x Ws with half-pixel centres, no antialiasing,
 *                           then /255, zero pad and HWC->CHW exactly as balf_preprocess_u8.
 * balf_merge_levels_topk    per-level keypoint lists (outputs of balf_windowed_nms_topk / balf_greedy_nms_topk at each
 *                           level, capacity K) -> the k_out best over all levels, ordered by (score descending, level
 *                           ascending, rank inside the level); coordinates mapped back to the level-0 frame:
 *                           x0 = (x + 0.5) * scale_x[level] - 0.5.  xy_out fp32 [B,k_out,2], score_out fp32 [B,k_out],
 *                           level_out int32 [B,k_out], count_out int32 [B].  xy / score / count are HOST arrays of
 *                           n_levels device pointers. */
#define BALF_MAX_LEVELS 8
BALF_API int balf_rgb_to_gray_u8(const uint8_t* rgb, int B, int H, int W, uint8_t* gray, void* stream);
BALF_API int balf_preprocess_f32(const float* img, int B, int H, int W, int C, float* x, int Hp, int Wp, int top, int left,
                                 void* stream);
BALF_API int balf_resize_preprocess_u8(const uint8_t* img, int B, int H, int W, int C, int Hs, int Ws, float* x, int Hp,
                                       int Wp, int top, int left, void* stream);
BALF_API int balf_merge_levels_topk(int n_levels, const int32_t* const* xy, const float* const* score,
                                    const int32_t* const* count, const float* scale_x, const float* scale_y, int B, int K,
                                    int k_out, float* xy_out, float* score_out, int32_t* level_out, int32_t* count_out,
                                    void* stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md section 8(f3): repeatability metrics and their homography helpers.  float64 throughout (the reference works
 * on Python floats); point arrays are [n,4] = (x, y, radius, score) unless stated.  Homographies are HOST arrays of 9
 * doubles (row-major 3x3).
 * balf_apply_homography_to_points  replaces balf/benchmark_test/geometry_tools.py:43-64 (+ getAff :66-84): positions through
 *     H, radii through the local affine approximation of H.
 * balf_common_region_masks         replaces geometry_tools.py:7-27 (create_common_region_masks): uint8 masks [src_h,src_w]
 *     and [dst_h,dst_w]; cv2.warpPerspective (INTER_LINEAR, 1/32-pixel grid, zero border) of border-masked ones, >= 0.75,
 *     border mask again.
 * balf_compute_repeatability       replaces balf/benchmark_test/repeatability_tools.py:379-490 (+ :492-513): scalars[8]
 *     (device) = rep_single_scale, rep_multi_scale, num_points_single_scale, num_points_multi_scale,
 *     error_overlap_single_scale, error_overlap_multi_scale, total_num_points, possible_matches; corr_s / corr_m
 *     int32 [min(n1,n2),2] = (index in dst, index in src) in the order the reference appends them.  *overflow (device)
 *     is set when more candidate pairs than the workspace holds (64 per point) reached the overlap threshold.
 * balf_resize_repeatability        replaces repeatability_tools.py:516-614 (compute_resize_repeatability): kp / wkp [n,3]
 *     = (row, col, prob), H maps (x, y) of the first image to the second; out6 (device) = repeatability,
 *     localization_err, common_src_num, common_dst_num, rep_src_num, rep_dst_num.  The inputs are not modified (the
 *     reference overwrites `keypoints` in place, :560-561).
 * Ties in every sort resolve in index order (the canonical rule of this library, SURVEY.md section 8c). */
BALF_API int balf_apply_homography_to_points(const double* pts, int n, const double* h_host, double* out, void* stream);
BALF_API int balf_common_region_masks(const double* h_dst_2_src_host, int src_h, int src_w, int dst_h, int dst_w, int border,
                                      uint8_t* mask_src, uint8_t* mask_dst, void* stream);
BALF_API size_t balf_repeatability_workspace_bytes(int n1, int n2);
BALF_API int balf_compute_repeatability(const double* src, int n1, const double* dst, int n2, double overlap_err, double eps,
                                        double dist_match_thresh, double radius_size, double* scalars, int32_t* corr_s,
                                        int32_t* corr_m, int32_t* overflow, void* workspace, size_t workspace_bytes,
                                        void* stream);
BALF_API int balf_resize_repeatability(const double* kp, int n1, const double* wkp, int n2, const double* h_host, int src_h,
                                       int src_w, int dst_h, int dst_w, int keep_k, double dist_thresh, double* out6,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Geometric verification of match lists: RANSAC homography, batched over image pairs.  No reference counterpart (the
 * reference stops at the SMNN matches; its HPatches / GoPro evaluation parsers name the measure without implementing it):
 * the semantics are defined here, restated in oracle/homography.py and checked against that restatement and against
 * cv2.findHomography(RANSAC).  float64 throughout, no fused multiply-add, so a result is a pure function of
 * (inputs, thr, iters, seed).
 * p1, p2 float64 [B,M,2] = (x, y) of the matches of each pair, count int32 [B] valid rows per pair (clamped to [0, M]).
 * Outputs: H float64 [B,9] (row-major, H[8] = 1) mapping p1 to p2, inlier_mask uint8 [B,M], n_inliers int32 [B].
 *  - Sampling: hypothesis h (0 <= h < iters) of pair b draws its 4 indices from
 *      stream = splitmix64(splitmix64(seed) ^ (b << 32 | h)),  index_c = splitmix64(stream + c) mod n,  c = 0, 1, ...
 *    (splitmix64(z): z += 0x9E3779B97F4A7C15; z = (z ^ z >> 30) * 0xBF58476D1CE4E5B9; z = (z ^ z >> 27) *
 *    0x94D049BB133111EB; z ^ z >> 31, all mod 2^64).  An index already in the sample is skipped; a hypothesis that has not
 *    found 4 distinct indices after 32 counters is degenerate.
 *  - Minimal solver: each image's 4 points are normalised to centroid 0 and mean distance sqrt(2) (sums in index order);
 *    the 8x8 DLT system with h33 = 1 is solved by Gaussian elimination with partial pivoting (first maximum wins); then
 *    H = T2^-1 Hn T1, scaled to H[8] = 1.  Degenerate (score -1): any 3 of the 4 points collinear in either image
 *    (|cross product of two triangle edges| <= 1e-6 in normalised coordinates, or not a number), a pivot that is 0 or not
 *    finite, or H[8] = 0 / not finite before the scaling.
 *  - Inliers: w = (H p1)_z > 0 and |(H p1)_xy * (1 / w) - p2|^2 <= thr^2 (squared distances, no square root).
 *    Score = inlier count; the winner of a pair is the highest score, the lowest h among equal scores.
 *  - Refit: the winner's inliers are refitted with the same normalised DLT through its 8x8 normal equations and the same
 *    elimination, the sums accumulated in a fixed order (oracle/homography.py restates it).  Each refit replaces H and its
 *    inliers; the refits repeat while the inlier count grows, at most 8 times.  The outputs are the last H and its inliers.
 *  - A pair with fewer than 4 matches or no non-degenerate hypothesis: H all zeros, n_inliers = 0, mask all zeros.
 * Argument errors (< 0): thr <= 0 (or NaN), iters outside [1, 131072], M outside [0, 16384] (test_utils.K_MAX),
 * B outside [0, 65535], a workspace smaller than balf_homography_workspace_bytes(B, M, iters). */
BALF_API size_t balf_homography_workspace_bytes(int B, int M, int iters);
BALF_API int balf_find_homography_ransac(const double* p1, const double* p2, const int32_t* count, int B, int M,
                                         double thr, int iters, uint64_t seed, double* H, uint8_t* inlier_mask,
                                         int32_t* n_inliers, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Geometric verification of match lists of general 3-D scenes: RANSAC fundamental matrix, batched over image pairs.  No
 * reference counterpart (its GoPro evaluation parser, config_gopro_eval.py, names the measure without implementing it):
 * the semantics are defined here, restated in oracle/fundamental.py and checked against that restatement and against
 * cv2.findFundamentalMat.  float64, no fused multiply-add, and only + - * / sqrt and comparisons, so a result is a pure
 * function of (inputs, thr, iters, seed).
 * Inputs and outputs use the homography's layouts: p1, p2 float64 [B,M,2], count int32 [B] (clamped to [0, M]); outputs
 * F float64 [B,9] (row-major) with x2^T F x1 = 0 (F maps p1 to epipolar lines in image 2), inlier_mask uint8 [B,M],
 * n_inliers int32 [B].
 *  - Sampling: the homography's hash streams unchanged (stream = splitmix64(splitmix64(seed) ^ (b << 32 | h)),
 *    index_c = splitmix64(stream + c) mod n), drawing 7 distinct indices; a hypothesis that has not found them after 64
 *    counters has no model.
 *  - Minimal solver (7-point): each image's 7 points normalised to centroid 0 and mean distance sqrt(2) (sums in index
 *    order); the 2-D null space {F1, F2} of the 7x9 system by the homography's partial-pivot elimination (F1: f8 = 1,
 *    f7 = 0; F2: f8 = 0, f7 = 1; a pivot that is 0 or not finite: no model); the real roots lam of
 *    det(lam F1 + (1 - lam) F2) = 0, a cubic whose roots are bracketed (its derivative's roots split the Cauchy bound
 *    interval into monotone pieces) and bisected, so up to 3 models per hypothesis, model m of hypothesis h in slot
 *    3 h + m; each model F = T2^T Fn T1.
 *  - Scaling: every F has unit Frobenius norm and its first largest-magnitude entry positive (cv2 divides by F[8] where it
 *    can; F is defined up to scale only).  A norm of 0 or not finite: no model.
 *  - Inliers: with l2 = F x1 = (a, b, c), s = x2^T F x1 and l1 = F^T x2 = (a', b', c'), a match is an inlier when
 *    s^2 <= thr^2 (a^2 + b^2) and s^2 <= thr^2 (a'^2 + b'^2), each a^2 + b^2 finite and > 0: both point-to-epipolar-line
 *    distances are at most thr (cv2's FM_RANSAC error, squared).  The winner is the highest count, the lowest 3 h + m among
 *    equal counts.
 *  - Refit: when the winner has at least 8 inliers, the normalised 8-point least squares on them: the eigenvector of the
 *    smallest eigenvalue of the 9x9 normal matrix (sums in the homography's fixed order) by cyclic Jacobi, made rank 2 in
 *    normalised coordinates as F - (F v3) v3^T (v3 from a 3x3 Jacobi of F^T F: the nearest rank-2 matrix), denormalised
 *    and scaled.  Each refit replaces F and its inliers; the refits repeat while the inlier count grows and is at least 8,
 *    at most 8 times.
 *  - A pair with fewer than 7 matches or no model: F all zeros, n_inliers = 0, mask all zeros.  With exactly 7 matches
 *    cv2 returns all (up to 3) solutions stacked; this runs RANSAC as usual and returns the best one.
 *  - Limits: plane degeneracy is not handled (no DEGENSAC).  On a planar scene (or a pure rotation) the returned F fits
 *    the matches but the epipolar geometry is not determined by them.
 * Argument errors (< 0): thr <= 0 (or NaN), iters outside [1, 131072], M outside [0, 16384], B outside [0, 65535], a
 * workspace smaller than balf_fundamental_workspace_bytes(B, M, iters). */
BALF_API size_t balf_fundamental_workspace_bytes(int B, int M, int iters);
BALF_API int balf_find_fundamental_ransac(const double* p1, const double* p2, const int32_t* count, int B, int M,
                                          double thr, int iters, uint64_t seed, double* F, uint8_t* inlier_mask,
                                          int32_t* n_inliers, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY.md section 8(e): the one collective of the sharded path.  No reference counterpart (the reference is single-device,
 * demo/demo_match.py:29): image batches are partitioned over the ranks, every rank runs the whole pipeline on its shard, and
 * the fixed-size keypoint records are all-gathered over NCCL (NVLink 5 / NVSwitch).
 * `comm` is an ncclComm_t; NCCL is bound at run time from the libnccl.so.2 the process already uses.  The helpers create
 * one from a 128-byte ncclUniqueId (host) that rank 0 obtains and the caller distributes by any means.
 * balf_gather_keypoints: xy int32 [B_local,K,2], score fp32 [B_local,K], count int32 [B_local] of this rank ->
 *     xy_all [world*B_local,K,2], score_all [world*B_local,K], count_all [world*B_local] in rank order, on every rank. */
BALF_API int balf_nccl_unique_id(void* id_host_128);
BALF_API int balf_nccl_comm_create(const void* id_host_128, int world, int rank, void** comm_out);
BALF_API int balf_nccl_comm_destroy(void* comm);
BALF_API size_t balf_gather_workspace_bytes(int world, int B_local, int K);
BALF_API int balf_gather_keypoints(void* comm, int world, const int32_t* xy, const float* score, const int32_t* count, int B_local,
                                   int K, int32_t* xy_all, float* score_all, int32_t* count_all, void* workspace,
                                   size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BALF_B200_H_ */
