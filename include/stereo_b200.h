/*
 * stereo_b200.h -- C ABI of libstereo_b200.so (sm_100a).
 *
 * Drop-in boundary for the Stereo R-CNN hot path.  Every entry point takes
 * plain device pointers + sizes + an explicit stream (a cudaStream_t passed
 * as void*), never allocates, never synchronises, and returns 0 on success
 * or a non-zero code (a cudaError_t value, or SB_EINVAL for a bad argument /
 * too-small workspace).  Caller allocates every output, as in the reference.
 *
 * Reference interfaces replaced (paths relative to the reference checkout):
 *   sb_nms                    <- lib/model/nms/src/nms_cuda_kernel.h:5-6  (nms_cuda_compute)
 *                                lib/model/nms/src/nms_cuda.h:4-5         (nms_cuda, THC glue)
 *   sb_roi_align_forward      <- lib/model/roi_align/src/roi_align_kernel.h:13-17 (ROIAlignForwardLaucher)
 *                                lib/model/roi_align/src/roi_align_cuda.h:1-2     (roi_align_forward_cuda)
 *   sb_roi_align_backward     <- lib/model/roi_align/src/roi_align_kernel.h:24-27 (ROIAlignBackwardLaucher)
 *                                lib/model/roi_align/src/roi_align_cuda.h:4-5     (roi_align_backward_cuda)
 *   sb_proposal_layer         <- lib/model/rpn/proposal_layer.py:42-145 (_ProposalLayer.forward)
 *   sb_dense_align            <- lib/model/dense_align/dense_align.py:240-300 (align_parallel)
 *   sb_roi_align_pyramid_nhwc <- lib/model/stereo_rcnn/stereo_rcnn.py:110-139 (PyramidRoI_Feat + RoIAlignAvg)
 *   sb_conv2d / sb_* layer ops<- torch.nn.Conv2d/BatchNorm2d/... call sites in
 *                                lib/model/stereo_rcnn/resnet.py:66-121,236-286 and
 *                                lib/model/rpn/stereo_rpn.py:32-40,73-95
 */
#ifndef STEREO_B200_H
#define STEREO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_OK 0
#define SB_EINVAL (-22)

typedef void* sb_stream_t; /* cudaStream_t */

/* library / device info: returns the compute capability major*10+minor of device 0, <0 on error */
int sb_version(void);
int sb_device_cc(void);

/* ---------------------------------------------------------------- NMS ----
 * dets: n x 5 [x1,y1,x2,y2,score] fp32, pre-sorted by score desc.
 * keep: >= n int32 (ascending indices of kept boxes), num_out: 1 int32.
 * Suppress j>i when IoU(i,j) > thresh ("+1" areas), bit-exact with the
 * reference's bitmask + greedy scan; the scan runs on the device.            */
size_t sb_nms_workspace_bytes(int n);
int sb_nms(const float* dets, int n, float thresh, int* keep, int* num_out,
           void* workspace, size_t workspace_bytes, sb_stream_t stream);
/* the raw 64x64 bitmask, upper-triangle blocks only (blocks below the diagonal are zero) */
int sb_nms_mask(const float* dets, int n, float thresh, uint64_t* mask, sb_stream_t stream);

/* ----------------------------------------------------------- RoIAlign ----
 * Reference semantics: features NCHW fp32, rois R x 5 [batch,x1,y1,x2,y2],
 * (ah, aw) is the tap lattice (RoIAlignAvg passes pooled+1), out R x C x ah x aw. */
int sb_roi_align_forward(const float* features, int N, int C, int H, int W,
                         const float* rois, int R, int ah, int aw, float spatial_scale,
                         float* out, sb_stream_t stream);
/* bottom_grad (N x C x H x W) must be zero-filled by the caller, as in the reference.
 * Like the reference kernel (roi_align_kernel.cu:94-143) the scatter uses four float
 * atomicAdds per tap: the summation ORDER is not deterministic, results agree with the
 * reference launcher to 1e-4 relative (tests/test_gpu_ops.py), not bit for bit.        */
int sb_roi_align_backward(const float* top_grad, int N, int C, int H, int W,
                          const float* rois, int R, int ah, int aw, float spatial_scale,
                          float* bottom_grad, sb_stream_t stream);

/* The same backward, deterministic (SURVEY 7.8): contributions are accumulated in 64-bit fixed point (scale from
 * max|top_grad|, quantum max|top| * 2^-41), so the sums do not depend on the order of the atomics or of the RoIs --
 * bit-identical run to run.  bottom_grad is OVERWRITTEN (no zero-fill needed); workspace = N*C*H*W*8 + 16 bytes. */
size_t sb_roi_align_backward_det_workspace(int N, int C, int H, int W);
int sb_roi_align_backward_det(const float* top_grad, int N, int C, int H, int W,
                              const float* rois, int R, int ah, int aw, float spatial_scale,
                              float* bottom_grad, void* workspace, size_t workspace_bytes, sb_stream_t stream);

/* Fused PyramidRoI_Feat: level routing (Q14) + per-level scale (Q15) + tap lattice +
 * 2x2/stride-1 average, NHWC features, one launch for all levels.
 * feats[l]: N x H_l x W_l x C (l = P2..P5); out[r][ph][pw][out_coff + c], row pitch out_ld elements;
 * round_tf32: 0 = exact fp32, 1 = fp32 rounded to TF32, 2 = __half output (out is then a __half*). */
int sb_roi_align_pyramid_nhwc(const float* const* feats, const int* heights, const int* widths,
                              int C, float im_h, const float* rois, int R, int pooled,
                              float* out, int out_ld, int out_coff, int round_tf32, sb_stream_t stream);

/* Exact adjoint of sb_roi_align_pyramid_nhwc (PyramidRoI_Feat, stereo_rcnn.py:110-139, whose backward is the
 * RoIAlignAvg autograd of modules/roi_align.py:26-29 -> roi_align_kernel.cu:94-143 per level): the same level routing,
 * per-level scale, (P+1)^2 lattice and 2x2 average, transposed.  top_grad[r][ph][pw][top_coff + c] (row pitch top_ld)
 * -> grad_feats[l] = N x H_l x W_l x C fp32, l = P2..P5, OVERWRITTEN.  Accumulated in 64-bit fixed point as
 * sb_roi_align_backward_det (quantum max|top_grad| * 2^-41, found on the device): the result does not depend on the
 * order of the atomics or of the RoIs -- bit-identical run to run.  C % 4 == 0.  A RoI whose batch index (column 0)
 * is outside [0, N) contributes nothing (the forward reads such a RoI's taps unchecked; the backward never writes
 * outside the feature gradients).                                                                                  */
size_t sb_roi_align_pyramid_nhwc_backward_workspace(int N, const int* heights, const int* widths, int C);
int sb_roi_align_pyramid_nhwc_backward(const float* top_grad, int top_ld, int top_coff, int C, float im_h,
                                       const float* rois, int R, int pooled, int N, const int* heights,
                                       const int* widths, float* const* grad_feats, void* workspace,
                                       size_t workspace_bytes, sb_stream_t stream);

/* ----------------------------------------------------- proposal layer ----
 * cls_prob [B,A,2] (column 1 = score), bbox_pred_lr [B,A,6], im_info [B,3] (device).
 * cfg: host struct (anchor pyramid + top-N / threshold constants), A = n_ratios*sum(h*w).
 * rois_left/right: [B, post_nms_top_n, 5], zero padded; fully stream-ordered.          */
typedef struct {
    int n_levels;             /* <= 8 */
    int shapes[8][2];         /* (h, w) of each pyramid level (rpn_shapes) */
    int anchor_scales[8];     /* cfg.FPN_ANCHOR_SCALES */
    int feat_strides[8];      /* cfg.FPN_FEAT_STRIDES  */
    int n_ratios;             /* <= 4 */
    double ratios[4];         /* cfg.ANCHOR_RATIOS */
    int pre_nms_top_n;        /* cfg[key].RPN_PRE_NMS_TOP_N  (<= 16384) */
    int post_nms_top_n;       /* cfg[key].RPN_POST_NMS_TOP_N */
    float nms_thresh;         /* cfg[key].RPN_NMS_THRESH */
} sb_proposal_cfg;
size_t sb_proposal_workspace_bytes(int B, int A, int pre_nms_top_n);
int sb_proposal_layer(const float* cls_prob, const float* bbox_pred_lr, const float* im_info,
                      int B, int A, const sb_proposal_cfg* cfg,
                      float* rois_left, float* rois_right,
                      void* workspace, size_t workspace_bytes, sb_stream_t stream);
/* the whole anchor table of the pyramid (generate_anchors.py:112-173: fp64, cast to fp32), [A,4] in the proposal
 * layer's order (level, y, x, ratio); only shapes / anchor_scales / feat_strides / ratios of cfg are read.  The
 * proposal layer itself never materialises it; the train-time anchor target layer (below) needs it. */
int sb_generate_anchors(const sb_proposal_cfg* cfg, int A, float* anchors, sb_stream_t stream);
/* fused RPN head epilogue: raw head output [B, sum(h*w), ld] (cols 0..5 cls logits in the
 * reference's channel order, 6..23 the 18 box channels) -> cls_prob [B,A,2], bbox_pred [B,A,6]
 * with the reference's softmax channel pairing (stereo_rpn.py:52-60,81-83)               */
int sb_rpn_head_epilogue(const float* head, int B, int P, int ld, float* cls_prob, float* bbox_pred,
                         sb_stream_t stream);

/* -------------------------------------------------------- dense_align ----
 * im_left/right: 3 x H x W planar fp32 (network-scale, batch 1).
 * calib4: host {P2[0,0], P2[0,2], P2[1,2], P2[0,3]-P3[0,3]}; scale = im_info[0,2].
 * box_left D x 4, keypoints D x 5, poses D x 7 (device).  status[D], best_dis[D] (device). */
size_t sb_dense_align_workspace_bytes(int H, int W, int D);
int sb_dense_align(const float* im_left, const float* im_right, int H, int W,
                   const double* calib4, double scale,
                   const float* box_left, const float* keypoints, const float* poses, int D,
                   float* status, float* best_dis,
                   void* workspace, size_t workspace_bytes, sb_stream_t stream);

/* ----------------------------------------------------- dense layer ops ----
 * NHWC fp32 activations.  One descriptor drives both the SIMT fp32 kernel (stem, odd
 * shapes) and the tcgen05 TF32 implicit-GEMM kernel (everything GEMM-shaped).          */
typedef struct {
    const float* in;        /* [N,H,W,in_ld] channels [0,Cin) used */
    const float* wgt;       /* [Cout][kh][kw][Cin] */
    const float* scale;     /* [Cout] or NULL (folded frozen BN gamma/sqrt(var+eps)); 16-byte aligned for the tcgen05 path */
    const float* shift;     /* [Cout] or NULL (folded BN beta / conv bias); 16-byte aligned for the tcgen05 path */
    const float* residual;  /* [N,Ho,Wo,res_ld] or NULL: added before ReLU (tcgen05 path: 1x1 convs only -- conv3 of a
                             * bottleneck; sb_conv2d_tc_supported() says no otherwise and the SIMT kernel takes it) */
    const float* up_src;    /* [N,UH,UW,Cout] or NULL: bilinear(align_corners) upsample to Ho x Wo, added */
    float* out;             /* out[n*out_n_stride + ho*out_h_stride + wo*out_w_stride + out_coff + c] */
    int N, H, W, Cin, Cout, kh, kw, stride, pad, Ho, Wo;
    int in_ld, res_ld, UH, UW, relu;
    int out_coff;
    /* TF32 operand hygiene (tcgen05 kind::tf32 TRUNCATES fp32 operands to 19 bits, a biased rounding):
     *   out_mode 0: store exact fp32 (tensors read by non-conv consumers)
     *   out_mode 1: store round-to-nearest TF32 (tensors read only by convs: truncation becomes exact)
     *   out_mode 2: store exact fp32 with +0x1000 added to the bit pattern ("pre-biased"): the tensor
     *               core's truncation then IS round-to-nearest, and exact readers subtract 0x1000 back
     *               (residual stream of the trunk: conv input and exact residual from one tensor)
     *   res_biased: the residual tensor is stored pre-biased;  in_biased: the input is (SIMT kernel only) */
    int out_mode, res_biased, in_biased;
    long long out_n_stride, out_h_stride, out_w_stride;
    /* fp16 operand mode of the tensor-core kernel (kind::f16, fp32 accumulate): in/wgt point to __half data
     * (in_dtype 1, Cin % 64 == 0); out16, when non-NULL, receives an fp16 (round-to-nearest) twin of the
     * output with the same element strides; out may be NULL when only the fp16 twin is wanted.          */
    void* out16;
    int in_dtype;
    int max_ctas;           /* 0 = one persistent CTA per SM; otherwise cap the grid (concurrent launches on
                             * other streams get the remaining SMs) */
} sb_conv_desc;

int sb_conv2d_simt(const sb_conv_desc* d, sb_stream_t stream);
/* tcgen05 path: requires Cin % 32 == 0 (K tile = one 128-byte swizzle row), stride 1. */
int sb_conv2d_tc(const sb_conv_desc* d, sb_stream_t stream);
int sb_conv2d_tc_supported(const sb_conv_desc* d);

/* Diagnostics (tools/conv_trace.py): per-CTA phase timestamps of every following sb_conv2d_tc launch, 16 x u64
 * per CTA and 304 CTA slots per launch, into a caller-owned device buffer of sb_conv_trace_bytes(max_launches)
 * bytes.  buf = NULL switches tracing off.  No counterpart in the reference. */
size_t sb_conv_trace_bytes(int max_launches);
int sb_conv_trace(void* buf, int max_launches);
int sb_conv_trace_count(void);
int sb_conv_trace_info(int id, int* out12);

/* GEMM on the tcgen05 tensor cores with operands read in their stored layout (the building block of the backward
 * passes: weight gradients contract over pixels / RoIs, data gradients multiply by the untransposed weight -- the
 * adjoints of the nn.Linear / 1x1 Conv2d products of resnet.py:256-263,282-285):
 *   C[m][n] = alpha * sum_k A(m,k) * B(n,k) + bias[n]
 * a, b: __half; a_mn_major = 0: A stored [M][lda], A(m,k) = a[m*lda + k];  1: stored [K][lda], A(m,k) = a[k*lda + m].
 *       b_mn_major = 0: B stored [N][ldb];  1: stored [K][ldb], B(n,k) = b[k*ldb + n].
 * c: fp32 [M][ldc] (overwritten).  alpha: DEVICE scalar or NULL (= 1), so that a scale computed on the device needs no
 * host read (graph capturable).  bias: fp32 [N] or NULL.  fp32 accumulation; any M, N, K >= 1; lda / ldb / ldc
 * multiples of 8 elements, a / b / c / bias 16-byte aligned (SB_EINVAL otherwise).  No split-K: C is bit-identical
 * from run to run.  No transposed copy of an operand is made.                                                      */
typedef struct {
    const void* a;
    const void* b;
    float* c;
    const float* alpha;
    const float* bias;
    int M, N, K;
    int lda, ldb, ldc;
    int a_mn_major, b_mn_major;
} sb_gemm_desc;
int sb_gemm_tc(const sb_gemm_desc* d, sb_stream_t stream);

/* stem: NCHW image -> conv7x7/2 + frozen BN + ReLU -> NHWC (resnet.py:111-113) */
int sb_stem_conv(const float* im_nchw, int N, int H, int W, const float* wgt /*[64][7][7][3]*/,
                 const float* scale, const float* shift, float* out_nhwc, int out_mode, sb_stream_t stream);
/* stem as a tensor-core GEMM: patch matrix [N*Ho*Wo][160] (k = ci*49+r*7+s, zero padded from 147) that
 * sb_conv2d_tc then multiplies with the [64][160] stem weights (1x1 conv, Cin = 160)              */
int sb_stem_im2col(const float* im_nchw, int N, int H, int W, float* out, sb_stream_t stream);
/* fp16 variant: rows of 152 __half (147 taps + 5 zeros; the GEMM multiplies them with [64][192] zero-padded weights,
 * the tensor map zero-fills columns 152..191 of the third 64-wide K-step) */
int sb_stem_im2col16(const float* im_nchw, int N, int H, int W, void* out_half, sb_stream_t stream);
/* the stem on the tensor cores with the patch gather INSIDE the GEMM kernel (round 2: no patch matrix in memory):
 * wgt16 = __half [64][192] ((ci, r, s) taps zero padded from 147), out16 = __half NHWC [N,Ho,Wo,64], BN + ReLU fused */
int sb_stem_conv_tc(const float* im_nchw, int N, int H, int W, const void* wgt16, const float* scale,
                    const float* shift, void* out16, sb_stream_t stream);
/* MaxPool2d(3, stride 2, pad 0, ceil_mode) NHWC (resnet.py:113) */
int sb_maxpool3x3s2_ceil(const float* in, int N, int H, int W, int C, float* out, sb_stream_t stream);
int sb_maxpool3x3s2_ceil16(const void* in_half, int N, int H, int W, int C, void* out_half, sb_stream_t stream);
/* x[:, ::2, ::2, :] (stride-2 1x1 convs of resnet.py:71 and P6 of stereo_rcnn.py:39) */
int sb_subsample2(const float* in, int N, int H, int W, int C, float* out, sb_stream_t stream);
/* keypoint tail: relu'd deconv output [R,G,G,C] -> sum over height -> 1x1 (C->6) -> [R,6,G]
 * -> softmax over 4G / G / G (stereo_rcnn.py:262-271)                                    */
int sb_kpts_tail(const void* x, int x_is_half, int R, int G, int C, const float* w /*[6][C]*/, const float* b /*[6]*/,
                 float* kpts_prob /*[R,4G]*/, float* left_prob /*[R,G]*/, float* right_prob /*[R,G]*/,
                 float* kpts_pred_all /*[R,6,G], required*/, sb_stream_t stream);
/* box-head tail: fc7 [R,K] -> cls softmax [R,nc], bbox [R,6nc], dim_orien [R,5nc] */
int sb_box_tail(const float* fc7, int R, int K, int n_classes,
                const float* w_cls, const float* b_cls, const float* w_box, const float* b_box,
                const float* w_dim, const float* b_dim,
                float* cls_prob, float* bbox_pred, float* dim_orien, sb_stream_t stream);
/* test-time decode (test_net.py:138-212), one image */
int sb_test_decode(const float* rois_left, const float* rois_right, const float* bbox_pred,
                   const float* dim_orien, const float* kpts_prob, const float* left_prob,
                   const float* right_prob, const float* im_info, int R, int n_classes, int grid,
                   float* pred_boxes_left, float* pred_boxes_right, float* dim_orien_out,
                   float* pred_kpts, sb_stream_t stream);
/* the same decode that also emits the per-image detection record which ranks all-gather (SURVEY 8e; the result
 * packing of test_net.py:233-330): record[r] = [cls_prob nc | boxes_left 4nc | boxes_right 4nc | dim_orien 5nc |
 * kpts 5], row pitch record_ld >= 14*nc + 5 floats                                                           */
int sb_test_decode_record(const float* rois_left, const float* rois_right, const float* cls_prob,
                          const float* bbox_pred, const float* dim_orien, const float* kpts_prob,
                          const float* left_prob, const float* right_prob, const float* im_info, int R,
                          int n_classes, int grid, float* pred_boxes_left, float* pred_boxes_right,
                          float* dim_orien_out, float* pred_kpts, float* record, int record_ld,
                          sb_stream_t stream);
/* per-class detection NMS (test_net.py:233-259), one image: scores [R,nc], boxes [R,4nc] (decoded left
 * boxes); keeps RoIs with score[:,cls] > score_thresh, sorted by score, NMS(nms_thresh); keep[] (>= R
 * ints) receives RoI indices in kept order, num_out the count.  R <= 512.                          */
int sb_class_nms(const float* scores, const float* boxes, int R, int n_classes, int cls,
                 float score_thresh, float nms_thresh, int* keep, int* num_out, sb_stream_t stream);
/* input pipeline (lib/model/utils/blob.py:44-64 prep_im_for_blob + demo.py:124-128): uint8 HWC image (BGR, or RGB
 * with rgb_input = 1 as scipy's imread returns it, demo.py:106) -> fp32 (pixel - cfg.PIXEL_MEANS) ->
 * cv2.resize(fx = fy = scale, INTER_LINEAR) -> out [3, Ho, Wo] CHW, (Ho, Wo) from sb_prep_image_size            */
int sb_prep_image_size(int H, int W, double scale, int* Ho, int* Wo);
int sb_prep_image(const uint8_t* img, int H, int W, double scale, int rgb_input, float* out, sb_stream_t stream);
/* L2 flush helper for benchmarks: writes `bytes` of scratch */
int sb_fill(float* p, size_t n, float v, sb_stream_t stream);
/* number of kernel launches issued by this library since load (bench "gpu_launches") */
unsigned long long sb_launch_count(void);

/* ------------------------------------------------- 3D box solvers (SURVEY 8f-1) ----
 * The CPU stage between the network and dense_align (test_net.py:262-325), on the device.
 * sb_infer_boundary: kitti_utils.infer_boundary (kitti_utils.py:398-437) over the kept detections (keep[0..*num),
 *   in kept order); boxes [R, ld] with the box at column col_offset; left_right [>= *num, 2].
 * sb_box_solve: the keypoint border fix-up (test_net.py:263-266, inferred may be NULL) and
 *   box_estimator.solve_x_y_z_theta_from_kpt (box_estimator.py:169-385) per kept detection of class `cls` with
 *   score > eval_thresh; solved detections are appended in order to boxes_all [cap,5] (box + score), kpts_all
 *   [cap,5], poses_all [cap,8] (x,y,z,w,h,l,theta,alpha) as test_net.py:281-303 builds them; src_index [cap] = RoI
 *   index, *n_out (device) = how many.  p2 / p3: 3x4 row-major projection matrices, (im_h, im_w) the ORIGINAL image.
 * sb_dense_align_n: sb_dense_align on those device-resident rows (count read on the device).
 * sb_box_rectify: box_estimator.solve_x_y_theta_from_kpt (box_estimator.py:387-545) with the aligned disparity ->
 *   final [cap,13] doubles: valid, score, box_left[4], x, y, z, w, h, l, theta (what write_detection_results takes).
 * The reference minimises with scipy Newton-CG; here Levenberg-Marquardt in fp64 on the same residuals, to a
 * tighter stationarity than Newton-CG's own end points (tests/test_box_solver.py).                              */
int sb_infer_boundary(const float* boxes, int ld, int col_offset, const int* keep, const int* num, int im_w,
                      float* left_right, sb_stream_t stream);
int sb_box_solve(const float* scores, const float* boxes_left, const float* boxes_right, const float* dim_orien,
                 const float* kpts, const int* keep, const int* num, const float* inferred, int n_classes, int cls,
                 int im_h, int im_w, const double* p2, const double* p3, float eval_thresh, int cap,
                 float* boxes_all, float* kpts_all, float* poses_all, int* src_index, int* n_out, sb_stream_t stream);
int sb_dense_align_n(const float* im_left, const float* im_right, int H, int W, const double* calib4, double scale,
                     const float* box_left, int box_ld, const float* keypoints, const float* poses, int pose_ld,
                     int D_cap, const int* n_dev, float* status, float* best_dis, void* workspace,
                     size_t workspace_bytes, sb_stream_t stream);
int sb_box_rectify(const float* boxes_all, const float* kpts_all, const float* poses_all, const float* succ,
                   const float* best_dis, const int* n, int cap, int im_h, int im_w, const double* p2,
                   const double* p3, double* final_out, sb_stream_t stream);

/* ------------------------------------------------- record all-gather over peer memory (SURVEY 8e) ----
 * The path's only exchange: every rank's fixed-size detection record ([300, 14nc+5] fp32, ~40 KB) to every rank of
 * one NVSwitch box.  Each rank owns a mailbox (sb_peer_alloc), exports it with CUDA IPC (sb_ipc_export, 64-byte
 * handle exchanged by the host's control plane) and maps its peers' (sb_ipc_import).  sb_peer_put_record stores the
 * local record into every mailbox (posted 128-bit NVLink writes + system-scope release of a sequence flag);
 * sb_peer_wait_records acquires the world's flags for the same step in the local mailbox and copies the records to
 * gathered[world][rec_floats].  Step counters live on the device: both calls are CUDA-graph capturable.  A peer
 * that never delivers sets *err_flag (device int) to 1 + its rank after timeout_s instead of hanging the GPU.
 * Replaces torch.distributed.all_gather / ncclAllGather on the data path; mailboxes[] is a HOST array of the
 * `world` device pointers (own allocation at index `rank`).                                                  */
size_t sb_peer_mailbox_bytes(int n_slots, int world, int rec_floats);
int sb_peer_alloc(size_t bytes, void** ptr);
int sb_peer_free(void* ptr);
int sb_ipc_export(void* ptr, void* handle64);
int sb_ipc_import(const void* handle64, void** ptr);
int sb_ipc_close(void* ptr);
int sb_peer_put_record(const float* rec, void* const* mailboxes, int n_slots, int world, int rec_floats,
                       int rank, int slot, sb_stream_t stream);
/* lag = 0: collect the step just put; lag = 1: collect the PREVIOUS step of this slot (pipelined exchange: no rank
 * waits for a slower peer's current step; the first call of a slot leaves `gathered` untouched) */
int sb_peer_wait_records(void* mailbox, int n_slots, int world, int rec_floats, int slot, int lag, float* gathered,
                         int* err_flag, double timeout_s, sb_stream_t stream);

/* ------------------------------------------------- train-time target layers and losses (SURVEY A16 / 8f-4) ----
 * The label / target assignment and the losses of one training step on the device, no host round trip.
 * Every compare is bit-identical to the reference (fp32, same operation order); the regression targets differ at most
 * in the last ulp of log().  The random sampler takes explicit words instead of numpy's global stream (which the
 * reference consumes with data-dependent lengths): see oracle/train_targets.py (NumpySampler / KeySampler).
 *
 * sb_anchor_targets -- _AnchorTargetLayer.forward (lib/model/rpn/anchor_target_layer.py:42-164):
 *   anchors [A,4] fp32 (all pyramid levels, the proposal layer's order), gt_left / gt_right / gt_merge [B,K,5]
 *   (x1, y1, x2, y2, class; zero rows pad to K <= 64), im_h / im_w = int(im_info[0][0..1]) (image 0 bounds the anchors
 *   of the whole batch, :70-73), keys [B,A] uint32: one random word per anchor -- when an image has more than
 *   num_fg foreground (or more than rpn_batchsize - n_fg background) anchors, those with the SMALLEST (key, index)
 *   are disabled, i.e. "the first n - keep of a random permutation" (:109-123).
 *   -> labels [B,A] (1 / 0 / -1), targets_left / targets_right [B,A,4] (bbox_transform_batch, bbox_transform.py:38-77;
 *   zeros outside the image), inside_w / outside_w [B,A] (outside = 1 / #sampled anchors of the LAST image, :136).
 * sb_proposal_targets -- _ProposalTargetLayer.forward (lib/model/rpn/proposal_target_layer.py:36-333):
 *   rois_left / rois_right [B,R,5] (batch index first), gt_* as above, gt_dim_orien [B,K,5], gt_kpts [B,K,6];
 *   keys [B,R+K] (one word per candidate incl. the appended ground-truth boxes: foreground = the fg_rois_per_image
 *   candidates with the smallest (key, index), in that order), words [B,S] (background draw j = candidate
 *   words[j] * n_bg >> 32, i.e. floor(u * n_bg) with u = words[j] / 2^32; also the with-replacement draws of the
 *   one-sided cases :249-265) -> S = rois_per_image rows per image: rois, labels, box targets (normalised),
 *   dimension / orientation targets, keypoint / border bin targets (int32) and weights, inside / outside weights,
 *   keep_inds (index into the R+K candidates) and status [B] (1 = neither foreground nor background, the
 *   reference's ValueError :267).  R + K <= 4096, S <= 1024.
 * sb_rpn_loss -- stereo_rpn.py:114-140: losses[0] = cross entropy over the anchors with label != -1, losses[1] =
 *   _smooth_l1_loss (net_utils.py:79-99, sigma 3) on the 6-d deltas; optional gradients w.r.t. rpn_cls_score [B,A,2] and
 *   rpn_bbox_pred [B,A,6] (both or neither), scaled by exp(-uncert[0..1]) when uncert != NULL.
 * sb_rcnn_loss -- stereo_rcnn.py:201-311: losses[0..3] = RCNN_loss_cls, RCNN_loss_bbox, RCNN_loss_dim_orien,
 *   RCNN_loss_kpts; bbox_pred [R,6C] / dim_orien_pred [R,5C] are the per-class outputs (gathered by label inside);
 *   optional gradients w.r.t. all six prediction tensors (all or none), scaled by exp(-uncert[2..5]).
 * sb_multitask_loss -- trainval_net.py:214-219: total = sum_i losses[i] exp(-uncert[i]) + uncert[i]; d_uncert optional.
 * sb_clip_gradient -- net_utils.clip_gradient (net_utils.py:37-49) over n_tensors gradient tensors (HOST arrays of
 *   device pointers / element counts): one global norm, one scale; norm_out [2] (device) = total norm, applied factor.
 * Reductions are two-level in a fixed order: deterministic.                                                     */
typedef struct sb_proposal_target_cfg {
    int rois_per_image;        /* cfg.TRAIN.BATCH_SIZE = 512                         */
    int fg_rois_per_image;     /* round(FG_FRACTION * BATCH_SIZE) = 128              */
    float fg_thresh;           /* 0.5                                                */
    float bg_thresh_hi;        /* 0.5                                                */
    float bg_thresh_lo;        /* 0.0                                                */
    float bbox_means[4];       /* BBOX_NORMALIZE_MEANS (0, 0, 0, 0)                  */
    float bbox_stds[4];        /* BBOX_NORMALIZE_STDS (0.1, 0.1, 0.2, 0.2)           */
    float dim_means[5];        /* DIM_NORMALIZE_MEANS (1.6, 1.5, 4.0, 0, 0)          */
    float dim_stds[5];         /* DIM_NORMALIZE_STDS (0.5 x 5)                       */
    int kpts_grid;             /* cfg.KPTS_GRID = 28                                 */
} sb_proposal_target_cfg;

size_t sb_anchor_targets_workspace(int B, int A);
int sb_anchor_targets(const float* anchors, int A, const float* gt_left, const float* gt_right,
                      const float* gt_merge, int B, int K, int im_h, int im_w, const unsigned* keys,
                      float neg_overlap, float pos_overlap, int rpn_batchsize, int num_fg, void* workspace,
                      size_t workspace_bytes, float* labels, float* targets_left, float* targets_right,
                      float* inside_w, float* outside_w, sb_stream_t stream);
int sb_proposal_targets(const float* rois_left, const float* rois_right, int B, int R, const float* gt_left,
                        const float* gt_right, const float* gt_dim_orien, const float* gt_kpts, int K,
                        const unsigned* keys, const unsigned* words, const sb_proposal_target_cfg* cfg,
                        float* out_rois_left, float* out_rois_right, float* labels, float* bbox_targets_left,
                        float* bbox_targets_right, float* dim_orien_targets, int* kpts_targets,
                        float* kpts_weight, float* inside_w, float* outside_w, int* keep_inds, int* status,
                        sb_stream_t stream);
size_t sb_loss_workspace_bytes(void);
int sb_rpn_loss(const float* rpn_cls_score, const float* rpn_bbox_pred, const float* labels,
                const float* targets_left, const float* targets_right, const float* inside_w,
                const float* outside_w, int B, int A, const float* uncert, void* workspace,
                size_t workspace_bytes, float* losses, float* d_cls_score, float* d_bbox_pred,
                sb_stream_t stream);
int sb_rcnn_loss(const float* cls_score, const float* bbox_pred, const float* dim_orien_pred,
                 const float* kpts_pred, const float* left_border_pred, const float* right_border_pred,
                 const float* labels, const float* bbox_targets_left, const float* bbox_targets_right,
                 const float* dim_orien_targets, const int* kpts_targets, const float* kpts_weight,
                 const float* inside_w, const float* outside_w, int R, int n_classes, int kpts_grid,
                 const float* uncert, float* losses, float* d_cls_score, float* d_bbox_pred,
                 float* d_dim_orien_pred, float* d_kpts_pred, float* d_left_border_pred,
                 float* d_right_border_pred, sb_stream_t stream);
int sb_multitask_loss(const float* losses, const float* uncert, int n, float* total, float* d_uncert,
                      sb_stream_t stream);
/* ------------------------------------------------- box-head training step (RCNN_top + tail, resnet.py:256-263,
 * 282-285,345-348; stereo_rcnn.py:248-257).  The fc6 / fc7 products and their adjoints run through sb_gemm_tc.
 * sb_dropout -- nn.Dropout(p = 0.2) after a ReLU with explicit random words (one uint32 per element, as the samplers
 *   above): out = x * 1.25 where words[i] >= 0.2 * 2^32, else 0; out32 and / or out16 (__half).
 * sb_box_tail_logits -- sb_box_tail writing the class LOGITS (the cross entropy of sb_rcnn_loss takes logits).
 * sb_box_tail_backward -- adjoint of the three tail linears: d_fc7 [R,K] = [d_cls|d_bbox|d_dim] [Wc;Wb;Wd], and the
 *   weight / bias gradients in the reference's shapes, fixed-order sums over R.
 * sb_dropout_backward -- g = dy * keep * 1.25 * (y > 0) (y = the ReLU output the dropout consumed), db [C] = sum_r g
 *   (fixed order; NULL: skipped), g16 = __half(g * 2^e) with e from max|g| on the device (largest element in
 *   [2^14, 2^15)), inv_scale [1] = 2^-e for sb_gemm_tc's alpha.  No host read.
 * sb_permute_pc_to_cp -- [Co][P][C] -> [Co][C][P] (the fc6 weight gradient from the GEMM's packed (ph, pw, c) order
 *   to Conv2d's [2048][512][7][7]).                                                                                */
int sb_dropout(const float* x, const unsigned* words, int R, int C, float* out32, void* out16, sb_stream_t stream);
int sb_box_tail_logits(const float* fc7, int R, int K, int n_classes,
                       const float* w_cls, const float* b_cls, const float* w_box, const float* b_box,
                       const float* w_dim, const float* b_dim,
                       float* cls_score, float* bbox_pred, float* dim_orien, sb_stream_t stream);
int sb_box_tail_backward(const float* d_cls, const float* d_bbox, const float* d_dim, const float* fc7, int R, int K,
                         int n_classes, const float* w_cls, const float* w_box, const float* w_dim, float* d_fc7,
                         float* dw_cls, float* db_cls, float* dw_box, float* db_box, float* dw_dim, float* db_dim,
                         sb_stream_t stream);
size_t sb_dropout_backward_workspace(int R, int C);
int sb_dropout_backward(const float* dy, const float* y, const unsigned* words, int R, int C, float* db, void* g16,
                        float* inv_scale, void* workspace, size_t workspace_bytes, sb_stream_t stream);
int sb_permute_pc_to_cp(const float* in, int Co, int P, int C, float* out, sb_stream_t stream);

size_t sb_clip_gradient_workspace(int n_tensors);
int sb_clip_gradient(float* const* grads, const size_t* counts, int n_tensors, float clip_norm,
                     void* workspace, size_t workspace_bytes, float* norm_out, sb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* STEREO_B200_H */
