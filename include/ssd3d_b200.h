/*
 * ssd3d_b200.h -- C ABI of libssd3d_b200.so: the sm_100a kernels behind the SSD3D detector hot path.
 *
 * The reference (Medical-Image-Analysis-Laboratory/MSLesions3D, lesions3d/) has no FFI of its own: the
 * path is a chain of torch calls.  Each entry point below replaces one such call site (cited as
 * file:line, relative to lesions3d/); the Python host in mslesions3d_b200/ binds them with ctypes and
 * keeps the reference's class/function surface (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; nothing here allocates or frees;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - return value: 0 on success, a cudaError_t (> 0) from the launch, or an SSD3D_ERR_* code (>= 10001);
 *   - activations are channels-last-3d (N, D, H, W, C) bf16; conv accumulation is fp32;
 *   - `nan_flag` (may be NULL) is a device int32 that kernels OR bits into instead of the reference's
 *     host-synchronising `isnan().sum() > 0` checks (mobilenet.py:46, ssd3d.py:95,258-261):
 *     bit 0 = backbone activation, bit 1 = locs, bit 2 = class scores.
 */
#ifndef SSD3D_B200_H_
#define SSD3D_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSD3D_OK 0
#define SSD3D_ERR_ARG 10001
#define SSD3D_ERR_TMA 10002
#define SSD3D_ERR_UNSUPPORTED 10003

#define SSD3D_NAN_BACKBONE 1
#define SSD3D_NAN_LOCS 2
#define SSD3D_NAN_SCORES 4

/* ------------------------------------------------------------------------------------------------
 * Prior (default) boxes as a closed-form function of the prior index (ssd3d.py:286-342, SURVEY.md 8f rank 3).
 * Prior p of layer l (start[l] <= p < start[l+1]):  local = p - start[l], b = local % n_boxes[l],
 * v = local / n_boxes[l], (i, j, k) = unravel(v, (d0, d1, d2)):
 *     cx = fp32((j + 0.5) / d1)   cy = fp32((i + 0.5) / d0)   cz = fp32((k + 0.5) / d2)     -- evaluated in
 * float64 and rounded once to fp32, exactly what the reference's Python doubles -> torch.FloatTensor do (note
 * the axis quirk: cx follows array axis 1, cy axis 0, ssd3d.py:304-309);  edge = size[l][b] three times, the
 * host-computed fp32(clamp(s + s/div, 0, 1)) of ssd3d.py:311,330.  Entry points whose name ends in _analytic
 * take a DEVICE copy of this table where their sibling takes the (P, 6) prior tensor, and recompute each prior
 * from its index instead of reading 24 bytes of it (60 MB per volume at 2.5 M priors); results are bit-identical.
 * ---------------------------------------------------------------------------------------------- */
#define SSD3D_MAX_PRIOR_LAYERS 8
#define SSD3D_MAX_PRIOR_SIZES 4
typedef struct ssd3d_prior_table {
  int32_t n_layers;
  int32_t d0[SSD3D_MAX_PRIOR_LAYERS], d1[SSD3D_MAX_PRIOR_LAYERS], d2[SSD3D_MAX_PRIOR_LAYERS];
  int32_t n_boxes[SSD3D_MAX_PRIOR_LAYERS];
  int32_t pad_;
  int64_t start[SSD3D_MAX_PRIOR_LAYERS + 1];
  float size[SSD3D_MAX_PRIOR_LAYERS][SSD3D_MAX_PRIOR_SIZES];
} ssd3d_prior_table;

/* Materialise the table: out (P, 6) fp32 = create_prior_boxes() (ssd3d.py:286-342).  table: device pointer. */
int ssd3d_prior_boxes(const ssd3d_prior_table* table, int64_t P, float* out, void* stream);

/* Library / build identification ("ssd3d_b200 sm_100a <n>"). */
const char* ssd3d_version(void);

/* ------------------------------------------------------------------------------------------------
 * Backbone (mobilenet.py:26-49, ssd3d.py:47-100)
 * ---------------------------------------------------------------------------------------------- */

/* Stem: dense Conv3d(Cin->Cout=32, k3, pad 1, stride (sd,2,2), no bias) + BN(eval, as scale/shift) + ReLU.
 * Replaces mobilenet.py:28-30 as instantiated at ssd3d.py:61.
 *   x      (N, Cin, D, H, W) NCDHW, fp32 (x_is_bf16 = 0, rounded to bf16 on load) or bf16; Cin in 1..4
 *   w      (32, KPAD) bf16, KPAD = 64 (Cin <= 2) or 128: the conv weight flattened as (Cout, Cin*27)
 *          -- PyTorch's own (Cout, Cin, 3,3,3) order -- zero padded along K
 *   scale, shift (32) fp32:  y = relu(conv * scale + shift)
 *   y      (N, Do, Ho, Wo, 32) bf16, Do = (D-1)/sd+1, Ho = (H-1)/2+1, Wo = (W-1)/2+1
 * Runs as a tcgen05 implicit GEMM fed by a 4-D TMA halo load when the row pitch W*elemsize is a multiple
 * of 16 bytes (ssd3d_stem_tc_supported), otherwise on the CUDA-core kernel (.._simt, same contract). */
int ssd3d_stem_conv_bn_relu(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift,
                            void* y, int N, int Cin, int D, int H, int W, int stride_d, void* stream);
int ssd3d_stem_conv_bn_relu_simt(const void* x, int x_is_bf16, const void* w, const float* scale,
                                 const float* shift, void* y, int N, int Cin, int D, int H, int W, int stride_d,
                                 void* stream);
int ssd3d_stem_tc_supported(int x_is_bf16, int Cin, int W);

/* One whole Block (mobilenet.py:34-49, eval mode) in ONE kernel: depthwise 3x3x3 + BN1 + ReLU -> pointwise 1x1x1 on
 * tcgen05 + BN2 + ReLU.  The depthwise tile (128 voxels x Cin, bf16, rounded exactly as the stand-alone kernel
 * stores it) stays in shared memory as the A operand of the pointwise GEMM, so the intermediate activation never
 * touches HBM.  Same arguments as ssd3d_dwconv3d_bn_relu followed by ssd3d_pwconv_bn_relu:
 *   x (N, D, H, W, Cin) bf16; w1 (27, Cin) bf16; w2 (Cout, Cin) bf16; scale / shift fp32; y (N, Do, Ho, Wo, Cout).
 * Built for the three large blocks of the backbone -- (Cin, Cout, stride) = (32, 64, 2), (64, 128, 2), (128, 128, 1)
 * on maps with Wo >= 8, Ho >= 4, Do >= 4 (ssd3d_block_fused_supported); other shapes return
 * SSD3D_ERR_UNSUPPORTED and the caller runs the two stand-alone kernels. */
int ssd3d_block_fused_supported(int Cin, int Cout, int D, int H, int W, int stride);
int ssd3d_block_dwpw_bn_relu(const void* x, const void* w1, const float* scale1, const float* shift1, const void* w2,
                             const float* scale2, const float* shift2, void* y, int N, int Cin, int Cout, int D, int H,
                             int W, int stride, int* nan_flag, void* stream);

/* Depthwise Conv3d(C, C, k3, pad 1, stride s in {1,2}, groups=C, no bias) + BN + ReLU.
 * Replaces mobilenet.py:38,44 (Block.conv1/bn1).
 *   x (N, D, H, W, C) bf16;  w (27, C) bf16, row = tap;  scale, shift (C) fp32;  C % 8 == 0
 *   y (N, Do, Ho, Wo, C) bf16 with Xo = (X-1)/s+1 */
int ssd3d_dwconv3d_bn_relu(const void* x, const void* w, const float* scale, const float* shift, void* y, int N,
                           int C, int D, int H, int W, int stride, void* stream);

/* Pointwise Conv3d(Cin->Cout, k1, no bias) + BN + ReLU as a tcgen05/TMEM GEMM with TMA-fed operands.
 * Replaces mobilenet.py:40,45 (Block.conv2/bn2) and the NaN check at mobilenet.py:46.
 *   x (M, Cin) bf16 (M = N*D*H*W rows of a channels-last activation);  w (Cout, Cin) bf16
 *   scale, shift (Cout) fp32;  y (M, Cout) bf16;  Cin % 32 == 0, Cout % 16 == 0 */
int ssd3d_pwconv_bn_relu(const void* x, const void* w, const float* scale, const float* shift, void* y,
                         int64_t M, int Cin, int Cout, int* nan_flag, void* stream);

/* SSD head for one feature map: loc conv and class conv (both k3, pad 1, with bias) fused into ONE
 * tcgen05 implicit GEMM whose epilogue writes straight into the concatenated outputs.
 * Replaces ssd3d.py:131-132,152-167 (two Conv3d + permute/contiguous/view + cat) and ssd3d.py:258-261.
 *   x      (N, D, H, W, C) bf16, C % 32 == 0
 *   w      (NPAD, 27*C) bf16, K index = tap*C + c; rows [0, bpl*6) = loc conv out channels, rows
 *          [bpl*6, bpl*(6+n_classes)) = class conv out channels, remaining rows zero; NPAD % 16 == 0
 *   bias   (NPAD) fp32
 *   locs   (N, P, 6) fp32, scores (N, P, n_classes) fp32; this layer writes priors
 *          [prior_offset, prior_offset + D*H*W*bpl) of every image, prior = ((d*H+h)*W+w)*bpl + b
 *   workspace: ssd3d_head_workspace_bytes(...) bytes (0 for large maps; small maps split K across CTAs and
 *          reduce partial sums in a fixed order)
 *   algo   0 = auto; 1 = per-tap TMA kernel (27 shifted 5-D boxes per chunk); 2 = halo-tile kernel (each
 *          activation voxel loaded once per 64-channel chunk, taps = row-shifted smem descriptors; needs
 *          C % 64 == 0 and NPAD <= 64); 3 = kw-GEMM + (kd,kh) stencil for maps with N*D*H*W >= 256 (
 *          C % 64 == 0, NPAD == 16): an implicit GEMM over the 3 W-taps with 144 output columns (9x the work
 *          per UMMA, 3 instead of 27 activation reads), then nine shifted reads per output from the L2-resident
 *          intermediate (in the workspace); 4 = the same with `w` ALREADY in the (144, 3*C) tiling produced by
 *          ssd3d_head_weight_kw (saves the per-call re-tiling when the weights are static, i.e. inference) */
int64_t ssd3d_head_workspace_bytes(int N, int C, int D, int H, int W, int NPAD);
int ssd3d_head_conv(const void* x, const void* w, const float* bias, float* locs, float* scores, int N, int C,
                    int D, int H, int W, int bpl, int n_classes, int NPAD, int64_t P, int64_t prior_offset,
                    int* nan_flag, void* workspace, int64_t workspace_bytes, int algo, void* stream);
/* (16, 27*C) packed head weight -> w_kw (144, 3*C) bf16: row (kd*3+kh)*16 + n, column kw*C + c.  C % 64 == 0 */
int ssd3d_head_weight_kw(const void* w, int C, void* w_kw, void* stream);
int ssd3d_head_kw_supported(int N, int C, int D, int H, int W, int NPAD);

/* ------------------------------------------------------------------------------------------------
 * Box geometry (utils.py:42-149).  All fp32, every arithmetic step separately rounded (no FMA).
 * ---------------------------------------------------------------------------------------------- */
#define SSD3D_BOX_CXCYCZ_TO_XYZ 0         /* utils.py:50-51   */
#define SSD3D_BOX_XYZ_TO_CXCYCZ 1         /* utils.py:101-102 */
#define SSD3D_BOX_GCXGCYGCZ_TO_CXCYCZ 2   /* utils.py:67-68   (needs priors) */
#define SSD3D_BOX_CXCYCZ_TO_GCXGCYGCZ 3   /* utils.py:88-89   (needs priors) */
int ssd3d_box_transform(int mode, const float* in, const float* priors, float* out, int64_t n, void* stream);

/* All-pairs intersection volume (want_iou = 0, utils.py:119-122) or Jaccard overlap (want_iou = 1,
 * utils.py:135-149) of boxes a (n1,6) and b (n2,6) in boundary coordinates -> out (n1, n2). */
int ssd3d_iou3d_pairwise(const float* a, const float* b, float* out, int64_t n1, int64_t n2, int want_iou,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Detection: softmax + decode + score filter + sort + greedy 3-D NMS + top-k  (ssd3d.py:344-460)
 * ---------------------------------------------------------------------------------------------- */

/* Bytes of scratch the detect call needs for the given problem (device memory, 256-byte aligned). */
int64_t ssd3d_detect_workspace_bytes(int N, int64_t P, int n_classes, int top_k);

/* One call = LSSD3D.detect_objects for the whole batch, no host synchronisation inside.
 *   locs (N,P,6), scores (N,P,n_classes) fp32 raw head outputs; priors (P,6) centre-size fp32
 *   min_score, max_overlap: thresholds already rounded to fp32 (strict > in both, ssd3d.py:388,422)
 *   Outputs, padded to top_k rows per image (rows >= out_count[i] are undefined):
 *     out_boxes (N, top_k, 6) fp32 boundary coords, out_scores (N, top_k) fp32,
 *     out_labels (N, top_k) int64, out_prior (N, top_k) int64 (prior index of each detection, -1 for
 *     the placeholder), out_count (N) int32.
 *   An image with no surviving box gets the reference's placeholder [0,0,0,1,1,1] / label 0 / score 0
 *   (ssd3d.py:437-440) and count 1.
 *   Tie rule for equal scores: ascending prior index (the stable order; the reference's sort is
 *   unspecified there, SURVEY.md M8).
 *   Any number of candidates is accepted: lists longer than SSD3D_SORT_MAX are reduced to their best
 *   10*top_k entries by a hierarchical block sort (exact).  Limit of this version: the NMS itself runs over
 *   at most min(10*top_k, SSD3D_SORT_MAX) boxes, and with P > SSD3D_SORT_MAX it needs 10*top_k <=
 *   SSD3D_SORT_MAX/2 (else SSD3D_ERR_UNSUPPORTED); bit 0 of *status (device int32, may be NULL) reports a
 *   truncated list. */
#define SSD3D_SORT_MAX 16384
int ssd3d_detect_objects(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                         int n_classes, float min_score, float max_overlap, int top_k, float* out_boxes,
                         float* out_scores, int64_t* out_labels, int64_t* out_prior, int32_t* out_count,
                         void* workspace, int64_t workspace_bytes, int32_t* status, void* stream);

/* Stage entry points (used by the stage-wise parity tests and by callers that want the pieces). */

/* softmax over classes + decode to boundary coords: probs (N, P, n_classes), boxes (N, P, 6). */
int ssd3d_decode_softmax(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                         int n_classes, float* probs, float* boxes_xyz, void* stream);

/* Greedy NMS over n boxes ALREADY sorted by descending score: keep (n) uint8, 1 = kept
 * (ssd3d.py:407-426).  mask_ws must hold n * ceil(n/64) uint64. */
int ssd3d_nms3d_sorted(const float* boxes_xyz, int64_t n, float max_overlap, uint8_t* keep, void* mask_ws,
                       void* stream);

/* Greedy NMS over a score-sorted list of ANY length (ssd3d.py:407-426 without the n x n IoU matrix, which
 * is 25 TB at the 2.5 M candidates of the whole-brain NMS-stress setting, model_insight.py:146): the list
 * is walked in chunks of `chunk` boxes (0 = default 4096; a multiple of 64 in [64, SSD3D_SORT_MAX]); each
 * chunk is first tested against the compact list of boxes kept so far, then resolved with the bit matrix.
 * With max_overlap >= 0 the cross test is pruned by a uniform grid over the boxes' minimum corners (only
 * intersecting boxes can suppress each other); SSD3D_NMS_NO_GRID in `flags` forces the dense cross test.
 * Same keep decisions as ssd3d_nms3d_sorted, bit for bit.  keep (n) uint8; kept_count (device int64, may
 * be NULL) receives the number of kept boxes; no host synchronisation.  chunk = 0: 4096 (the measured
 * optimum from 64 k to 2.5 M candidates). */
#define SSD3D_NMS_NO_GRID 1
int64_t ssd3d_nms3d_chunked_workspace_bytes(int64_t n, int chunk);
int ssd3d_nms3d_sorted_chunked(const float* boxes_xyz, int64_t n, float max_overlap, uint8_t* keep,
                               int64_t* kept_count, void* workspace, int64_t workspace_bytes, int chunk,
                               int flags, void* stream);

/* Ascending stable sort of n 64-bit keys in place (`Tensor.sort` of ssd3d.py:397,450 on the packed
 * {~orderable(score), index} keys, for lists the single-block sort cannot hold): 16384-key block sorts +
 * merge passes.  tmp: n keys of scratch (may be NULL when n <= SSD3D_SORT_MAX). */
int ssd3d_sort_keys_u64(uint64_t* keys, int64_t n, uint64_t* tmp, void* stream);

/* Stage 1 of detect_objects alone (ssd3d.py:363-388): softmax, decode to boundary coords, keep candidates
 * with score > min_score.  boxes_xyz (N,P,6); segment seg = img*(n_classes-1) + (c-1) owns
 * cand[seg*P .. seg*P + count[seg]) = keys {~orderable(score) << 32 | prior index} in arbitrary order;
 * count (N*(n_classes-1)) int32 is zeroed by the call. */
int ssd3d_decode_filter(const float* locs, const float* scores, const float* priors, int N, int64_t P,
                        int n_classes, float min_score, float* boxes_xyz, uint64_t* cand, int32_t* count,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training: prior <-> ground-truth matching and the MultiBox loss (ssd3d.py:741-941)
 * ---------------------------------------------------------------------------------------------- */

/* Matching + labelling + target encoding for a batch (ssd3d.py:786-888).
 *   gt_boxes (T, 6) fp32 boundary coords, all images concatenated; gt_labels (T) int64;
 *   gt_offsets (N+1) int32 prefix offsets (image i owns [gt_offsets[i], gt_offsets[i+1])), T = total
 *   priors_cxcycz (P, 6); thresholds t0 <= t1 (hard mode: t0 == t1), fp32-rounded
 *   true_classes (N, P) int64 in {-1, 0, 1..}; true_locs (N, P, 6) fp32
 *   overlap (N,P) fp32 and object_for_prior (N,P) int32: per-prior best IoU / object after the
 *   force-match; prior_for_object (T) int32: first-max prior of each object (ssd3d.py:811)
 *   best_key_ws: T * 8 bytes of scratch.  Images with no object are all background with zero targets
 *   (ssd3d.py:854-855).  Tie rules: first maximum (torch.max), last writer wins in the force-match. */
int ssd3d_match_priors(const float* gt_boxes, const int64_t* gt_labels, const int32_t* gt_offsets, int N,
                       int64_t T, const float* priors_cxcycz, int64_t P, float t0, float t1,
                       int64_t* true_classes, float* true_locs, float* overlap, int32_t* object_for_prior,
                       int32_t* prior_for_object, void* best_key_ws, void* stream);

/* MultiBox loss forward + analytic backward (ssd3d.py:891-941).
 *   out_loss (2) fp32 = {conf_loss, loc_loss}; n_pos_out (1) int32
 *   grad_locs (N,P,6), grad_scores (N,P,n_classes): d(conf_loss + alpha*loc_loss)/d input, may be NULL
 *   hard_negative_mining = 0 reproduces the shipped loss (all negatives, ssd3d.py:933); = 1 the
 *   commented variant (ssd3d.py:926-932) with neg_pos_ratio.
 *   workspace: ssd3d_multibox_workspace_bytes(N, P). */
int64_t ssd3d_multibox_workspace_bytes(int N, int64_t P);
int ssd3d_multibox_loss(const float* locs, const float* scores, const int64_t* true_classes,
                        const float* true_locs, int N, int64_t P, int n_classes, float alpha,
                        int hard_negative_mining, int neg_pos_ratio, float* out_loss, int32_t* n_pos_out,
                        float* grad_locs, float* grad_scores, void* workspace, int64_t workspace_bytes,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training step of the network (LSSD3D.training_step, ssd3d.py:467-531): what torch autograd derives for
 * the reference from nn.Conv3d / nn.BatchNorm3d / nn.ReLU (mobilenet.py:26-49, ssd3d.py:131-167) and
 * torch.optim.Adam (ssd3d.py:704-722).  Activations and activation gradients: channels-last bf16;
 * parameter gradients and optimizer state: fp32.  All reductions are two-stage and run-to-run reproducible.
 * ---------------------------------------------------------------------------------------------- */

/* Convolutions with an explicit epilogue y = conv * scale + shift, optional ReLU (relu = 0: identity).
 * relu = 1 is exactly the *_bn_relu entry point; training-mode BatchNorm needs the raw conv output
 * (scale = 1, shift = 0, relu = 0), and the pointwise data gradient dx = dz . W is the same GEMM with the
 * transposed weight. */
int ssd3d_stem_conv_affine(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift,
                           void* y, int N, int Cin, int D, int H, int W, int stride_d, int relu, void* stream);
int ssd3d_stem_conv_affine_simt(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift,
                                void* y, int N, int Cin, int D, int H, int W, int stride_d, int relu, void* stream);
/* The same stem contract on the banded-B tcgen05 kernel (csrc/conv_stem_tz.cu): the W taps live in a Toeplitz B
 * operand, the A operand is the raw TMA'd input row (no per-voxel tap gather), 512 voxels per accumulator, epilogue
 * straight to global memory.  bf16 volumes, Cin <= 2, W % 8 == 0 (ssd3d_stem_tz_supported);
 * ssd3d_stem_conv_affine / .._bn_relu pick it by themselves when it applies (SSD3D_STEM_TZ=0 turns that off). */
int ssd3d_stem_conv_affine_tz(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift,
                              void* y, int N, int Cin, int D, int H, int W, int stride_d, int relu, void* stream);
int ssd3d_stem_tz_supported(int x_is_bf16, int Cin, int W);
/* Stem + the depthwise conv of the first Block in ONE kernel (csrc/conv_stem_dw.cu; mobilenet.py:28-30 followed by
 * mobilenet.py:38,44 in eval mode): the stem activation (32 channels at half resolution, the largest tensor of the
 * network) stays in shared memory.  x as for the stem (bf16 only), w_stem (32, KPAD) bf16, w_dw (27, 32) bf16,
 * scale/shift = the two folded BatchNorms, y (N, Dd, Hd, Wd, 32) bf16 with Dd = ((D-1)/sd+1 - 1)/2 + 1 etc.
 * ssd3d_stem_dw_fused_supported: bf16 volumes, Cin <= 2, W = 128, even stem map along D and H. */
int ssd3d_stem_dw_fused(const void* x, int x_is_bf16, const void* w_stem, const float* scale0, const float* shift0,
                        const void* w_dw, const float* scale1, const float* shift1, void* y, int N, int Cin, int D,
                        int H, int W, int stride_d, void* stream);
int ssd3d_stem_dw_fused_supported(int x_is_bf16, int Cin, int D, int H, int W, int stride_d);
/* The gather-based tcgen05 stem kernel (csrc/conv_stem_tc.cu) addressed explicitly: the kernel ssd3d_stem_conv_affine
 * uses for fp32 volumes and Cin > 2; SSD3D_ERR_UNSUPPORTED when ssd3d_stem_tc_supported says no. */
int ssd3d_stem_conv_affine_tc(const void* x, int x_is_bf16, const void* w, const float* scale, const float* shift,
                              void* y, int N, int Cin, int D, int H, int W, int stride_d, int relu, void* stream);
int ssd3d_dwconv3d_affine(const void* x, const void* w, const float* scale, const float* shift, void* y, int N, int C,
                          int D, int H, int W, int stride, int relu, void* stream);
/* The depthwise entry points pick the TMA halo-tile kernel (conv_dw_tma.cu: one 5-D cp.async.bulk.tensor per
 * 32-channel tile, double buffered, persistent CTAs) for maps with Wo >= 8 and C % 32 == 0, else the direct
 * kernel (16-byte loads through L1); .._direct forces the latter (same contract; parity tests cover both). */
int ssd3d_dwconv3d_affine_direct(const void* x, const void* w, const float* scale, const float* shift, void* y, int N,
                                 int C, int D, int H, int W, int stride, int relu, void* stream);
int ssd3d_pwconv_affine(const void* x, const void* w, const float* scale, const float* shift, void* y, int64_t M,
                        int Cin, int Cout, int relu, int* nan_flag, void* stream);

/* BatchNorm3d in training mode + ReLU on a raw conv output z (M, C) bf16 (mobilenet.py:29-30,39,41,44-45):
 * batch mean / biased variance per channel -> scale = gamma/sqrt(var+eps), shift = beta - mean*scale
 * (fp32, C each; also mean and invstd for the backward), running statistics updated in place with
 * `momentum` and the unbiased variance (NULL to skip), *num_batches_tracked += 1 (device int64, NULL to skip),
 * a = relu(z*scale + shift) (NULL to skip).
 * workspace: ssd3d_bn_workspace_bytes(C). */
int64_t ssd3d_bn_workspace_bytes(int C);
int ssd3d_bn_train_fwd(const void* z, int64_t M, int C, const float* gamma, const float* beta, float eps,
                       float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                       float* scale, float* shift, float* mean, float* invstd, void* a, int* nan_flag,
                       void* workspace, int64_t workspace_bytes, void* stream);
/* Backward of the same unit: grad_a (M, C) bf16 = dL/da -> dgamma, dbeta (C) fp32 and dz (M, C) bf16
 * (dz may alias grad_a).  The ReLU mask is recomputed from z with the forward's arithmetic. */
int ssd3d_bn_relu_bwd(const void* z, const void* grad_a, int64_t M, int C, const float* scale, const float* shift,
                      const float* mean, const float* invstd, float* dgamma, float* dbeta, void* dz, void* workspace,
                      int64_t workspace_bytes, void* stream);
/* The same two passes as ONE launch each (csrc/bn_unit.cu): column sums, cross-CTA finalize and the elementwise
 * apply are phases of ONE grid -- thread-block clusters with distributed-shared-memory sums for maps up to 8192 rows,
 * (row chunk x channel group) tiles with one barrier per channel group above.  Arguments as
 * above plus `sync_words`: 512 device uint32, zero before the first launch, private to the calling stream (the
 * kernels leave them zero).  ssd3d_bn_unit_supported: 1 if (M, C) can take this path (C a multiple of 8; above 8192 rows a
 * multiple of 32, or C/8 a power of two in [4, 512]); workspace: ssd3d_bn_unit_workspace_bytes(C).  Replaces the same reference lines
 * (nn.BatchNorm3d + ReLU in train mode and their autograd backward, mobilenet.py:29-30,44-45). */
int ssd3d_bn_unit_supported(int64_t M, int C);
int64_t ssd3d_bn_unit_workspace_bytes(int C);
int ssd3d_bn_unit_fwd(const void* z, int64_t M, int C, const float* gamma, const float* beta, float eps,
                      float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                      float* scale, float* shift, float* mean, float* invstd, void* a, int* nan_flag,
                      void* workspace, int64_t workspace_bytes, uint32_t* sync_words, void* stream);
int ssd3d_bn_unit_bwd(const void* z, const void* grad_a, int64_t M, int C, const float* scale, const float* shift,
                      const float* mean, const float* invstd, float* dgamma, float* dbeta, void* dz, void* workspace,
                      int64_t workspace_bytes, uint32_t* sync_words, void* stream);

/* Weight gradients, dW = dz^T . im2col(x), split over rows and reduced in a fixed order.
 * workspace: ssd3d_wgrad_workspace_bytes(M, n_out, K) with (n_out, K) = (Cout, Cin) pointwise,
 * (16, 27*C) head, (32, 27*Cin) stem. */
int64_t ssd3d_wgrad_workspace_bytes(int64_t M, int n_out, int K);
/* pointwise: dz (M, Cout) bf16, x (M, Cin) bf16 -> dw (Cout, Cin) fp32.  Cin % 32 == 0, Cout % 64 == 0 */
int ssd3d_pwconv_wgrad(const void* dz, const void* x, int64_t M, int Cin, int Cout, float* dw, void* workspace,
                       int64_t workspace_bytes, void* stream);
/* stem: dz (N, Do, Ho, Wo, 32) bf16, x (N, Cin, D, H, W) fp32|bf16 -> dw (32, Cin, 3, 3, 3) fp32 */
int ssd3d_stem_wgrad(const void* dz, const void* x, int x_is_bf16, int N, int Cin, int D, int H, int W, int stride_d,
                     float* dw, void* workspace, int64_t workspace_bytes, void* stream);
/* stem unit backward without materialising dz (autograd of mobilenet.py:26-31 for the first layer, whose input needs
 * no gradient): after ssd3d_bn_unit_bwd(..., dz = NULL, ...) has left dgamma / dbeta, the BatchNorm + ReLU backward
 * is applied to grad_a (N, Do, Ho, Wo, 32) bf16 from the saved raw conv output z while the weight-gradient kernel
 * loads its rows.  Same result, bit for bit, as ssd3d_bn_unit_bwd + ssd3d_stem_wgrad.  SSD3D_ERR_UNSUPPORTED for
 * shapes the TMA tile kernel does not take (fewer than 128*148 output voxels, rows TMA cannot address). */
int ssd3d_stem_wgrad_bn(const void* z, const void* grad_a, const void* x, int x_is_bf16, int N, int Cin, int D, int H,
                        int W, int stride_d, const float* scale, const float* shift, const float* mean,
                        const float* invstd, const float* dgamma, const float* dbeta, float* dw, void* workspace,
                        int64_t workspace_bytes, void* stream);
/* head: dO (G, N*D*H*W, 16) bf16 gradient rows in G = ceil((n_loc+n_cls)/16) column groups
 * (ssd3d_head_grad_pack), x (N, D, H, W, C) bf16 -> dw_loc (n_loc, C, 3,3,3), dw_cls (n_cls, C, 3,3,3) fp32
 * (ssd3d.py:131-132: any n_classes).  One 16-column contraction pass per group.  C % 64 == 0, n_loc + n_cls <= 256 */
int ssd3d_head_wgrad(const void* dO, const void* x, int N, int C, int D, int H, int W, int n_loc, int n_cls,
                     float* dw_loc, float* dw_cls, void* workspace, int64_t workspace_bytes, void* stream);

/* Head gradient rows of one feature map from d(loss)/d(locs (N,P,6)), d(loss)/d(scores (N,P,n_classes)):
 * dO (G, N*D*H*W, 16) bf16, G = ceil(n_cols/16) groups of 16 columns in the column order of the fused head GEMM
 * ([loc | class | zero pad], n_cols = bpl*(6+n_classes) <= 256), and the bias gradients dbias_loc (bpl*6),
 * dbias_cls (bpl*n_classes) fp32 (column sums of the fp32 values).
 * workspace: ssd3d_head_grad_workspace_bytes(N, D, H, W, n_cols). */
int64_t ssd3d_head_grad_workspace_bytes(int N, int D, int H, int W, int n_cols);
int ssd3d_head_grad_pack(const float* dlocs, const float* dscores, int N, int D, int H, int W, int bpl,
                         int n_classes, int64_t P, int64_t prior_offset, void* dO, float* dbias_loc, float* dbias_cls,
                         void* workspace, int64_t workspace_bytes, void* stream);
/* Head data gradient (transposed 3x3x3 conv): dx (N, D, H, W, C) bf16 = conv_transpose(dO, w) + addend
 * (addend: the gradient arriving from the next backbone block, may be NULL, may alias dx).
 * dO (G, N*D*H*W, 16) as above; w: the packed head weight (16*G, 27*C) bf16 of ssd3d_head_conv; n_cols =
 * bpl*(6+n_classes).  C % 64 == 0 */
int ssd3d_head_dgrad(const void* dO, const void* w, const void* addend, void* dx, int N, int C, int D, int H, int W,
                     int n_cols, void* stream);

/* Depthwise 3x3x3 backward: dz (N, Do, Ho, Wo, C) bf16, w (27, C) bf16, x (N, D, H, W, C) bf16
 * -> dx (N, D, H, W, C) bf16;  dw (C, 1, 3, 3, 3) fp32.  workspace: ssd3d_dw_wgrad_workspace_bytes(C). */
int ssd3d_dwconv3d_dgrad(const void* dz, const void* w, void* dx, int N, int C, int D, int H, int W, int stride,
                         void* stream);
int64_t ssd3d_dw_wgrad_workspace_bytes(int C);
int ssd3d_dwconv3d_wgrad(const void* dz, const void* x, int N, int C, int D, int H, int W, int stride, float* dw,
                         void* workspace, int64_t workspace_bytes, void* stream);

/* Analytic-prior siblings (see ssd3d_prior_table above): identical contracts and bit-identical results, with a
 * device pointer to the prior table where the sibling takes the (P, 6) prior tensor
 * (ssd3d_decode_softmax / ssd3d_decode_filter / ssd3d_detect_objects: ssd3d.py:344-460;
 * ssd3d_match_priors: ssd3d.py:786-888). */
int ssd3d_decode_softmax_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table, int N,
                                  int64_t P, int n_classes, float* probs, float* boxes_xyz, void* stream);
int ssd3d_decode_filter_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table, int N,
                                 int64_t P, int n_classes, float min_score, float* boxes_xyz, uint64_t* cand,
                                 int32_t* count, void* stream);
int ssd3d_detect_objects_analytic(const float* locs, const float* scores, const ssd3d_prior_table* table, int N,
                                  int64_t P, int n_classes, float min_score, float max_overlap, int top_k,
                                  float* out_boxes, float* out_scores, int64_t* out_labels, int64_t* out_prior,
                                  int32_t* out_count, void* workspace, int64_t workspace_bytes, int32_t* status,
                                  void* stream);
int ssd3d_match_priors_analytic(const float* gt_boxes, const int64_t* gt_labels, const int32_t* gt_offsets, int N,
                                int64_t T, const ssd3d_prior_table* table, int64_t P, float t0, float t1,
                                int64_t* true_classes, float* true_locs, float* overlap, int32_t* object_for_prior,
                                int32_t* prior_for_object, void* best_key_ws, void* stream);

/* One Adam step over flat fp32 buffers with torch.optim.Adam's arithmetic (L2 weight decay added to the
 * gradient, bias-corrected moments; ssd3d.py:716): elements [0, bias_start) use lr, [bias_start, n) use
 * lr_bias (the reference's "biases at 2x lr" group, ssd3d.py:715).  grad is multiplied by grad_scale first
 * (1/world_size after the NCCL sum).  step >= 1.
 * status (2 int32, may be NULL): a step whose gradient holds a NaN / Inf (a batch without any positive prior
 * makes the MultiBox loss 0/0; the reference raises "Loss is NaN", ssd3d.py:938-940) is SKIPPED -- parameters and
 * moments untouched -- with status[0] = 1 for this call and status[1] incremented; status[1] must be zeroed once
 * by the caller.  After an all-reduce every rank sees the same non-finite values, so all ranks skip together. */
int ssd3d_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                    int64_t bias_start, float lr, float lr_bias, float beta1, float beta2, float eps,
                    float weight_decay, int step, float grad_scale, int32_t* status, void* stream);

/* The same step with its whole state on the device, so that forward .. backward .. all-reduce .. optimizer can be
 * ONE captured CUDA graph (no host scalar changes between replays): state (4 int32, zeroed once by the caller) =
 * {non-finite flag of this step, skipped steps, APPLIED steps, unused}; scalars (8 fp32 scratch).  The applied-step
 * counter k drives both the bias correction and the reference's CosineAnnealingLR(T_max = t_max), stepped once
 * per batch before the optimizer step (ssd3d.py:525-527, 718-720): lr_k = base_lr * (1 + cos(pi*k/t_max)) / 2
 * (t_max = 0: constant base_lr); biases use lr_k * bias_lr_mult (ssd3d.py:715).  A step with a non-finite gradient
 * is skipped and advances neither the counter nor the schedule (the reference raises and applies no step). */
int ssd3d_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                        int64_t bias_start, float base_lr, float bias_lr_mult, int t_max, float beta1, float beta2,
                        float eps, float weight_decay, float grad_scale, int32_t* state, float* scalars, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Detection metrics of ONE class (utils.py:155-230 compute_metrics_per_class + the cumulative precision /
 * recall / 11-point AP of utils.py:296-318), called from training_step / validation_step (ssd3d.py:499-518,
 * 563-584) and predict.py:279-281.  No host synchronisation.
 *   det_boxes (nd,6) boundary coords, det_scores (nd), det_images (nd) int32: image index of each detection
 *   true_boxes (nt,6), true_difficulties (nt) uint8, true_images (nt) int32
 *   recall_thresholds (n_thresholds <= 16) fp32 (the reference: torch.arange(0, 1.1, .1))
 * Outputs, detections in descending score order (equal scores: ascending input index):
 *   sorted_scores (nd), sort_index (nd) int32 (input index of each sorted position),
 *   true_positives / false_positives (nd) fp32 in {0,1}, detected (nt) uint8, true_volumes (nt) fp32,
 *   cum_precision / cum_recall (nd), out_stats (4 + n_thresholds) = {AP, recall, precision, F1, precision at
 *   every threshold}.   workspace: ssd3d_map_workspace_bytes(nd, nt).  nd >= 1. */
int64_t ssd3d_map_workspace_bytes(int64_t nd, int64_t nt);
int ssd3d_map_class(const float* det_boxes, const float* det_scores, const int32_t* det_images, int64_t nd,
                    const float* true_boxes, const uint8_t* true_difficulties, const int32_t* true_images, int64_t nt,
                    float min_overlap, const float* recall_thresholds, int n_thresholds, float* sorted_scores,
                    int32_t* sort_index, float* true_positives, float* false_positives, uint8_t* detected,
                    float* true_volumes, float* cum_precision, float* cum_recall, float* out_stats, void* workspace,
                    int64_t workspace_bytes, void* stream);

/* dst[i] = src[index[i]] (0 where index[i] < 0), converted to bf16 (dst_is_bf16 = 1) or kept fp32: every packed
 * weight layout of the step (stem (32,KPAD), depthwise (27,C), pointwise and its transpose, head (16,27*C) and
 * its bias) produced from the flat fp32 parameter buffer in one launch after the optimizer step. */
int ssd3d_gather_cast(const float* src, const int32_t* index, int64_t n, void* dst, int dst_is_bf16, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Input preparation (SURVEY.md 8f rank 2): MONAI NormalizeIntensity(nonzero=True) of the data module
 * (datasets.py:403) on the device.  x: `items` = N*C contiguous volumes of `voxels` fp32 values (NCDHW);
 * per item z-score over the non-zero voxels (population std; std == 0 -> 1; zeros stay zero), written as fp32 or
 * bf16 in the same layout -- the stem's input format.  workspace: ssd3d_normalize_workspace_bytes(items).
 * ---------------------------------------------------------------------------------------------- */
int64_t ssd3d_normalize_workspace_bytes(int items);
int ssd3d_normalize_intensity_nonzero(const float* x, int items, int64_t voxels, void* y, int y_is_bf16,
                                      void* workspace, int64_t workspace_bytes, void* stream);

/* Synthetic lesion volumes on the device (SURVEY.md 8f rank 2; generate_artificial_dataset.py:63-105): per volume
 * first_idx + n uniform noise in [0, 1) per channel, randint(num_lo, num_hi) + 1 cubes of side
 * randint(size_lo, size_hi) at corner randint(0, dim - side) per axis (shared by the channels), each adding 0.4 and
 * clipping to [0, 1], and the binary mask of the cubes.  Every value is a pure function of (seed, volume index,
 * channel, voxel) through Philox4x32-10 (the reference's serial MT19937 stream is NOT reproduced; same
 * distribution, same construction; restated in numpy by oracle/philox_oracle.py).
 *   out_raw (N, C, D, H, W) fp32 raw intensities (feed ssd3d_normalize_intensity_nonzero for datasets.py:403)
 *   mask    (N, D, H, W) uint8, may be NULL      (feed ssd3d_gt_boxes_from_segmentation for utils.py:438-513)
 *   cubes   (N, max_cubes, 4) int32 {side, corner d, h, w}, n_cubes (N) int32;  max_cubes <= 64 */
int ssd3d_generate_volumes(uint64_t seed, int64_t first_idx, int N, int C, int D, int H, int W, int num_lo,
                           int num_hi, int size_lo, int size_hi, int max_cubes, float* out_raw, uint8_t* mask,
                           int32_t* cubes, int32_t* n_cubes, void* stream);

/* Ground-truth boxes from segmentation volumes (SURVEY.md 8f rank 2; utils.py:438-513 BoundingBoxesGeneratord,
 * segmentation_mode "binary" (n_classes = 0: every non-zero voxel, label 1) or "classes" (n_classes >= 1: voxels
 * equal to c in 1..n_classes, label c; classes = [1..n_classes] as datasets.py:405 passes them)).
 * seg: (N, D, H, W) uint8 (seg_dtype 0) or fp32 (seg_dtype 1).  Per volume: face-connected components
 * (scipy.ndimage.label's default structure) per class, one box [min d, min h, min w, max d, max h, max w] /
 * [D, H, W, D, H, W] (inclusive max index, fp32 division) per component, in the reference's order: class
 * ascending, then the component's first voxel in C order; components one voxel thick along an axis have zero
 * volume and are dropped (utils.py:475-480).
 *   boxes (N, max_boxes, 6) fp32, labels (N, max_boxes) int64: rows [0, counts[n]) are valid
 *   n_components (N): components found before the zero-volume filter; a value > max_boxes means the lists
 *   were truncated and must not be used.  (The reference's c*1000 instance ids cap a class at 999 components.)
 * ---------------------------------------------------------------------------------------------- */
int64_t ssd3d_gt_boxes_workspace_bytes(int N, int D, int H, int W, int max_boxes);
int ssd3d_gt_boxes_from_segmentation(const void* seg, int seg_dtype, int N, int D, int H, int W, int n_classes,
                                     int max_boxes, float* boxes, int64_t* labels, int32_t* counts,
                                     int32_t* n_components, void* workspace, int64_t workspace_bytes, void* stream);

/* The same for segmentation_mode "instances" (utils.py:439-441,483-513): the volume holds one integer id per
 * object; thresholds (device int32 [n_thresholds][2]) map the id range [min_c, max_c) to class c+1.  One box per
 * id over ALL its voxels, ordered by class, then ascending id (np.unique); ids outside every range, non-integer
 * values and ids >= id_limit are ignored; ranges must not overlap.  Same outputs and zero-volume filter as
 * above; n_components = ids that fell into a range. */
int64_t ssd3d_gt_boxes_instances_workspace_bytes(int N, int id_limit, int max_boxes);
int ssd3d_gt_boxes_from_instances(const void* seg, int seg_dtype, int N, int D, int H, int W,
                                  const int32_t* thresholds, int n_thresholds, int id_limit, int max_boxes,
                                  float* boxes, int64_t* labels, int32_t* counts, int32_t* n_components,
                                  void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training from a device-resident data set: sampling and augmentation inside the captured training step.
 *
 * ssd3d_augment_batch builds one training batch in one launch.  Slot b takes subject
 * order[(step * N * world + rank * N + b) mod S] (DistributedSampler's split; the last batch wraps around, so
 * every batch holds N volumes).  Its draws come from Philox4x32-10, key = seed, counter = (rank * N + b, draw
 * counter low, draw counter high, call), with u01(u) = (u >> 8) * 2^-24, Bernoulli(p) = u01 < p and
 * randint(lo, hi) = lo + ((u * (hi - lo)) >> 32) as ssd3d_generate_volumes:
 *   call 0 {positive crop, box, rot90, k}, call 1 {offset d, h, w}, call 2 {flip d, h, w}, call 3 {scale, shift}.
 * Applied in this order, to the image and the mask alike:
 *   1. crop to (d, h, w): with probability pos_ratio, if the subject has a lesion box, one of its boxes
 *      (uniform) and per axis an offset uniform over the windows that contain the box -- or, on an axis where the
 *      box is longer than the window, its centre voxel (lo + hi) / 2; otherwise uniform over [0, src - out].
 *   2. np.rot90(x, k, axes = (rot_axis0, rot_axis1)) with probability rot90_prob, k uniform in {1, 2, 3}; the
 *      two output extents must be equal.
 *   3. np.flip of each spatial axis with probability flip_prob.
 *   4. (image only) y = bf16_rn(fp32_rn(fp32_rn(x * fp32_rn(1 + f)) + o)), f = scale * (2 u01 - 1),
 *      o = shift * (2 u01 - 1), per volume and shared by its channels (MONAI's non-channel-wise default).
 * Bounding boxes of the mask follow from it through ssd3d_gt_boxes_from_segmentation (utils.py:438-513).
 *   src (S, C, Ds, Hs, Ws) fp32 (src_is_bf16 = 0) or bf16; masks (S, Ds, Hs, Ws) uint8; order (S) int32
 *   state (8 int64) = {seed, draw counter, step in the epoch, rank, world size, 0 (kernel scratch), -, -}: the
 *         launch advances the draw counter and the step by one, so a captured graph draws a new batch per replay
 *   boxes (B, 6) int32 lesion boxes in voxel indices [lo d, lo h, lo w, hi d, hi h, hi w] (inclusive), subject s
 *         owning rows [box_offsets[s], box_offsets[s + 1])
 *   out (N, C, d, h, w) bf16, out_mask (N, d, h, w) uint8, record (N, 16) int32 = {subject, offset d, h, w, k,
 *         flip d, h, w, positive crop, box (-1: none), f (fp32 bits), o (fp32 bits), step, draw counter low,
 *         global slot, boxes of the subject}.
 * d, h, w <= Ds, Hs, Ws; w % 16 == 0 (16-byte stores); probabilities in [0, 1].
 *
 * ssd3d_gt_pack turns the per-image output of ssd3d_gt_boxes_from_segmentation (boxes (N, max_boxes, 6), labels
 * (N, max_boxes), counts, n_components) into the packed ground truth of the training step: gt_boxes
 * (N * per_volume, 6), gt_labels (N * per_volume) int64 and offsets (N + 1) int32 (the ssd3d_match_priors input),
 * without a host sync.  A batch in which a volume has more boxes than per_volume, or more components than
 * max_boxes (its list was truncated), overflows: it is packed as a batch without ground truth -- no positive
 * prior, so the MultiBox gradient is non-finite and ssd3d_adam_step_dev skips and counts the step -- and
 * status (2 int32) = {overflow of this batch, overflowing batches so far} records it (status[1] zeroed once by
 * the caller).  N <= 8192. */
int ssd3d_augment_batch(const void* src, int src_is_bf16, const uint8_t* masks, int S, int C, int Ds, int Hs, int Ws,
                        const int32_t* order, int64_t* state, const int32_t* boxes, const int32_t* box_offsets, int N,
                        int d, int h, int w, float pos_ratio, float flip_prob, float rot90_prob, int rot_axis0,
                        int rot_axis1, float scale, float shift, void* out, uint8_t* out_mask, int32_t* record,
                        void* stream);
int ssd3d_gt_pack(const float* boxes, const int64_t* labels, const int32_t* counts, const int32_t* n_components,
                  int N, int max_boxes, int per_volume, float* gt_boxes, int64_t* gt_labels, int32_t* offsets,
                  int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSD3D_B200_H_ */
