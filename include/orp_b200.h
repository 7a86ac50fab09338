/*
 * orp_b200.h - C ABI of liborp_b200.so: the B200 (sm_100a) implementation of the
 * OrientedRepPoints dense-inference hot path (SURVEY.md section 8).
 *
 * Plain pointers and sizes only - no torch types.  Every entry point cites the reference
 * interface it replaces.  Two families:
 *
 *   *_host   : host buffers in / host buffers out, blocking - drop-in for the reference's
 *              own C entry points that Cython binds (DOTA_devkit/poly_nms_gpu/*.hpp).
 *   (others) : DEVICE pointers, asynchronous on `stream` (a cudaStream_t passed as void*),
 *              what the reference's pybind11 torch extensions (mmdet/ops/.../src/*_cuda.cpp)
 *              do with at::Tensor::data_ptr().  Scratch memory comes from the CUDA
 *              stream-ordered pool (cudaMallocAsync) of the current device.
 *
 * All functions return 0 on success, a negative ORP_E* code otherwise; orp_last_error()
 * gives the message (thread-local).  There is no CPU fallback anywhere in this library.
 */
#ifndef ORP_B200_H_
#define ORP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORP_OK 0
#define ORP_EINVAL (-1)   /* bad argument                                  */
#define ORP_ECUDA (-2)    /* CUDA runtime error (see orp_last_error)        */
#define ORP_ENOGPU (-3)   /* no sm_100 device / wrong architecture          */
#define ORP_EOVERFLOW (-4) /* internal capacity exceeded after retries       */

const char *orp_last_error(void);
/* library/ABI version (major*100+minor) and the SM architecture it was compiled for (100) */
int orp_version(void);
int orp_compiled_sm(void);
/* number of kernel launches issued by this library since load / since the last reset
 * (bench.py reports it as "gpu_launches") */
int64_t orp_launch_count(void);
void orp_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Rotated / polygon NMS
 * ---------------------------------------------------------------------------------------- */

/* IoU arithmetic used to decide `iou > thr`:
 *   ORP_NMS_EXACT64  candidate pairs from an exact-safe AABB sweep; fp32 convex clipping in
 *                    pair-local coordinates with a proven error band; pairs inside the band are
 *                    re-evaluated with the reference's fp64 algorithm (DOTA_devkit/polyiou.cpp)
 *                    so every decision equals the fp64 reference decision.  Default.
 *   ORP_NMS_COMPAT32 the reference's fp32 arithmetic (mmdet/ops/nms/src/rnms_kernel.cu:17-147),
 *                    origin-anchored triangle fan, every pair of the upper triangle evaluated,
 *                    no operation contracted - bit-identical to mmdet/ops/nms/src/rnms_cpu.cpp.
 */
#define ORP_NMS_EXACT64 0
#define ORP_NMS_COMPAT32 1

/* degenerate-union convention:
 *   ORP_UNION_NAN_KEEPS      rnms  (rnms_kernel.cu:131-147: 0/0 = NaN, `NaN > thr` false)
 *   ORP_UNION_GUARD          poly_gpu_nms (poly_nms_kernel.cu:205-210: (inter+1)/(union+1))
 *   ORP_UNION_NAN_SUPPRESSES py_cpu_nms_poly (ResultMerge.py:39 keeps only `iou <= thr`)
 */
#define ORP_UNION_NAN_KEEPS 0
#define ORP_UNION_GUARD 1
#define ORP_UNION_NAN_SUPPRESSES 2

/* output ordering of the kept indices:
 *   ORP_ORDER_INDEX_ASC  rnms_cuda (rnms_kernel.cu:261-264)
 *   ORP_ORDER_SCORE_DESC poly_gpu_nms (poly_nms.pyx:19-24), py_cpu_nms_poly (ResultMerge.py:28-41)
 */
#define ORP_ORDER_INDEX_ASC 0
#define ORP_ORDER_SCORE_DESC 1

/* Greedy rotated NMS over n quadrilaterals, optionally segmented.
 *   dets      device float32 [n, 9] rows (x1,y1,x2,y2,x3,y3,x4,y4,score), row stride 9
 *   segments  device int32 [n] or NULL: boxes only interact inside one segment (class id for
 *             multiclass_rnms - replaces the coordinate-offset trick of
 *             mmdet/core/post_processing/bbox_nms.py:156-158; (image,class) id for ResultMerge)
 *   keep_out  device int64 [n]: kept original row indices, in `order`
 *   num_out   device int32 [1]: number kept
 * Replaces rnms_cuda() (mmdet/ops/nms/src/rnms_kernel.cu:204-265, bound at
 * mmdet/ops/nms/src/rnms_cuda.cpp:8-17).  Ties in score: lower row index first.
 * iou_thr is a double because the fp64 reference compares against a Python float
 * (ResultMerge.py:39); COMPAT32 rounds it to fp32 like rnms_cuda's `float nms_overlap_thresh`.
 * Asynchronous; nothing is copied to the host (one exception: if the candidate-pair list
 * outgrows its first allocation the call synchronises once and retries with the exact size). */
int orp_rnms(const float *dets, const int32_t *segments, int n, double iou_thr, int iou_mode,
             int union_mode, int order, int64_t *keep_out, int32_t *num_out, void *stream);

/* Drop-in for `void _poly_nms(int* keep_out, int* num_out, const float* polys_host,
 * int polys_num, int polys_dim, float nms_overlap_thresh, int device_id)`
 * (DOTA_devkit/poly_nms_gpu/poly_nms.hpp:9-10).  The reference's caller sorts polys_host by score
 * descending first (poly_nms.pyx:19-21) and gets positions in that order; this entry orders by score
 * itself (ties: lower row first), so sorted input gives exactly those positions and unsorted input gives
 * the same boxes as original row indices - the host sort can be dropped.
 * Host buffers, blocking.  polys_dim must be 9.  Unlike the reference, device_id is honoured. */
int orp_poly_nms_host(int *keep_out, int *num_out, const float *polys_host, int polys_num,
                      int polys_dim, float nms_overlap_thresh, int device_id);

/* Statistics of the last orp_rnms call on this thread.  Requires the stream to be synchronised by
 * the caller first. */
typedef struct {
    int64_t pairs_total;     /* pairs visited by the x-sweep (same segment, x-intervals overlap)  */
    int64_t pairs_aabb;      /* pairs whose axis-aligned hulls overlap                            */
    int64_t pairs_clipped;   /* pairs actually clipped: only (undecided box, KEPT candidate) pairs */
    int64_t pairs_fp64;      /* of those, decided by the fp64 reference algorithm (error band)    */
    int64_t edges;           /* candidate pairs: survivors of the exact-safe bounds (EXACT64), or
                                pairs with iou > thr (COMPAT32, where every pair is evaluated)    */
    int64_t suppressing;     /* clipped pairs with iou > thr                                      */
    int32_t overflow;        /* 1: the candidate list outgrew its buffer in a no-sync call        */
    int32_t rounds;          /* resolution rounds                                                */
    int32_t n;
} orp_nms_stats;
int orp_rnms_last_stats(orp_nms_stats *out);

/* Measurement hooks: with timing on, orp_rnms brackets its dominant kernel (the sweep+clip
 * kernel) with CUDA events ON THE LAUNCHING STREAM; orp_rnms_last_sweep_ms waits for them and
 * returns the elapsed device time of that kernel for the last call of this thread. */
void orp_set_timing(int on);
int orp_rnms_last_sweep_ms(float *ms);
/* with timing on, every tensor-core convolution launch is bracketed the same way; this collects (and
 * resets) the summed device time, the number of launches and their algorithmic FLOPs (2*MACs) since
 * the previous collect on this thread */
int orp_tc_timing_collect(float *total_ms, int *launches, double *flops);

/* ------------------------------------------------------------------------------------------
 * Pairwise rotated IoU
 * ---------------------------------------------------------------------------------------- */

/* Drop-in for `void _overlaps(float* overlaps, const float* boxes, const float* query_boxes,
 * int n, int k, int device_id)` (DOTA_devkit/poly_nms_gpu/poly_overlaps.hpp:1): (cx,cy,w,h,theta)
 * boxes -> corners as RotBox2Poly (poly_overlaps_kernel.cu:280-297) -> N x K IoU with the
 * zero-union guard (:300-328).  Host buffers, blocking. */
int orp_poly_overlaps_host(float *overlaps, const float *boxes, const float *query_boxes, int n,
                           int k, int device_id);
/* same on device pointers, asynchronous */
int orp_poly_overlaps(const float *boxes5, int n, const float *query5, int k, float *out,
                      void *stream);

/* N x K IoU of quadrilaterals (8 coords each), device pointers.  mode ORP_NMS_EXACT64 gives
 * fp32 values within 1e-5 of DOTA_devkit/polyiou.cpp (uncertain pairs recomputed in fp64);
 * ORP_NMS_COMPAT32 gives rnms_kernel.cu:131-147 bit-for-bit. */
int orp_quad_iou_matrix(const float *quads_a, int n, const float *quads_b, int k, int iou_mode,
                        int union_mode, float *out, void *stream);

/* fp64 IoU of aligned pairs with the algorithm and arithmetic of iou_poly()
 * (DOTA_devkit/polyiou.cpp:108-128) - the batched device equivalent of the SWIG call. */
int orp_iou_poly_f64_pairs(const double *p8, const double *q8, int n, double *out, void *stream);

/* IoU between the convex hull of each 9-point set and each quadrilateral: pts18 [N,18] (x0,y0,...,x8,y8),
 * quads8 [K,8] -> out [N,K] fp32, device resident.  Replaces convex_iou_cuda
 * (mmdet/ops/iou/src/convex_iou_kernel.cu:268-360; python side mmdet/ops/iou/iou_wrapper.py:21-30 convex_iou /
 * convex_overlaps).  fp64 gift-wrapping hull + fp64 polygon clipping as in the reference, float result. */
int orp_convex_iou(const float *pts18, int n, const float *quads8, int k, float *out, void *stream);

/* detectron2-style rotated boxes (cx,cy,w,h,theta in RADIANS as modified at
 * mmdet/ops/box_iou_rotated/src/box_iou_rotated_utils.h:59-62) -> N x M IoU; replaces
 * box_iou_rotated_cuda (box_iou_rotated_cuda.cu:13-62). */
int orp_box_iou_rotated(const float *boxes1, int n, const float *boxes2, int m, float *out,
                        void *stream);

/* ------------------------------------------------------------------------------------------
 * minaerarect
 * ---------------------------------------------------------------------------------------- */

/* 9-point sets -> minimum-area rectangles.  Replaces minareabbox_cuda()
 * (mmdet/ops/minarearect/src/minarearect_kernel.cu:470-505, bound at minarearect_cuda.cpp:5-13).
 *   pts       device float32 [n,18] rows (x0,y0,...,x8,y8), contiguous
 *   out       device float32 [n,8] corners (xmax,ymin),(xmin,ymin),(xmin,ymax),(xmax,ymax) of the
 *             winning rotated frame mapped back (kernel.cu:380-450)
 *   hull_map  device int32 [n,9] or NULL: hull vertex -> input point index, -1 padded
 *             (points_to_convex_ind, kernel.cu:330-340)
 *   scale, center: if center != NULL the fused affine of orientedreppoints_head.py:748-749 is
 *             applied: out = rect*scale + (center[2i],center[2i+1]) repeated 4 times; center is
 *             device float32 [n,2].  Pass scale=1, center=NULL for the bare op.
 * Asynchronous, output stays on the device (the reference copies through the host). */
int orp_minarearect(const float *pts, int n, float *out, int32_t *hull_map, float scale,
                    const float *center, void *stream);

/* ------------------------------------------------------------------------------------------
 * Head post-processing
 * ---------------------------------------------------------------------------------------- */

/* OrientedRepPointsHead.get_bboxes + multiclass_rnms for a whole batch, device resident
 * (mmdet/models/anchor_heads/orientedreppoints_head.py:673-779,
 *  mmdet/core/post_processing/bbox_nms.py:93-182).
 *   cls[l]   device fp32 NHWC [B, H[l], W[l], num_cls] logits (sigmoid classification)
 *   ref[l]   device fp32 NHWC [B, H[l], W[l], 18] refined points, (dy,dx) interleaved, stride units
 *   scale_factor  device fp32 [B] or NULL (= 1): boxes and points are divided by it (rescale=True)
 *   dets_out   device fp32 [B, max_per_img, 27] rows = reppoints(18) | box(8) | score, zero padded
 *   labels_out device int64 [B, max_per_img] (0-based class, -1 padding);  counts_out device int32 [B]
 * Per level top-k(nms_pre) on the max class score (ties: lower location first), class-aware NMS by
 * segment id instead of the coordinate-offset trick of bbox_nms.py:156-158, survivors in candidate
 * order unless more than max_per_img survive, then the max_per_img best by score.  Asynchronous. */
int orp_head_postprocess(int nlevels, const float *const *cls, const float *const *ref, const int *H,
                         const int *W, const int *stride, int B, int num_cls, int nms_pre, float score_thr,
                         double iou_thr, int max_per_img, const float *scale_factor, float *dets_out,
                         int64_t *labels_out, int32_t *counts_out, void *stream);
/* padded detections of orp_head_postprocess -> the fixed-layout payload of the ONE all-gather that replaces
 * collect_results_gpu (mmdet/apis/test.py:117-147): packed_out device fp32 [B, max_per_img + 1, 28], rows = 27 detection values |
 * label, zero padded; row max_per_img carries the image's count in column 0. */
int orp_pack_detections(const float *dets, const int64_t *labels, const int32_t *counts, int B, int max_per_img,
                        float *packed_out, void *stream);
/* orientedreppoints_head.py:162-163 for up to 8 pyramid levels in one launch: off = (1 - g) * pts + g * pts - base[c],
 * pts / off fp32 [.., 18] (host arrays of device pointers, element counts), base18 = the 3x3 grid (dy,dx) of :82-88 (host) */
int orp_dcn_offsets_multi(int nprob, const float *const *pts, float *const *off, const long long *numel,
                          float gradient_mul, const float *base18, void *stream);

/* ------------------------------------------------------------------------------------------
 * Dense layers, fp32 (CUDA cores) - the parity arithmetic of the backbone / FPN / head
 * All activations are NHWC ("channels last") contiguous device tensors; weights are
 * [Cout][KH][KW][Cin] (the reference's [Cout][Cin][KH][KW] permuted once at load time).
 * ---------------------------------------------------------------------------------------- */

/* y = relu?( conv(x, w) + bias + residual ), optionally accumulating the GroupNorm statistics of y:
 * gn_stats is device double [N, groups, 2] (sum, sum of squares), must be zeroed by the caller.
 * Replaces nn.Conv2d / ConvModule.conv (mmdet/ops/conv_module.py:124-132) on the cuDNN path; with
 * eval-mode BatchNorm folded into w and bias beforehand (the fold of tools/fuse_conv_bn.py:10-24). */
int orp_conv2d_f32(const float *x, int N, int H, int W, int Cin, const float *w, int Cout, int KH, int KW,
                   int stride, int pad, const float *bias, const float *residual, int relu, float *y,
                   double *gn_stats, int groups, void *stream);

/* Deformable convolution forward (DCNv1; DCNv2 when mask != NULL), deformable_groups = groups = 1.
 * Replaces deform_conv_forward_cuda / modulated_deform_conv_cuda_forward
 * (mmdet/ops/dcn/src/deform_conv_cuda.cpp:152-260, 490-569) without the im2col `columns` scratch:
 * sampling per deformable_im2col_bilinear (deform_conv_cuda_kernel.cu:84-115), validity test of :229.
 *   offset  device float32 [N, Ho, Wo, 2*KH*KW], channel 2t = dy, 2t+1 = dx of tap t (:222-225)
 *   mask    device float32 [N, Ho, Wo, KH*KW] or NULL */
int orp_deform_conv2d_f32(const float *x, int N, int H, int W, int Cin, const float *offset, const float *mask,
                          const float *w, int Cout, int KH, int KW, int stride, int pad, int dilation,
                          const float *bias, int relu, float *y, void *stream);

/* GroupNorm apply: y = relu?( (x - mean) * rstd * gamma + beta ) (+ nearest-2x upsampled up_src,
 * the FPN top-down add of mmdet/models/necks/fpn.py:150-154).  stats as produced by orp_conv2d_f32;
 * biased variance and eps as torch.nn.GroupNorm (mmdet/ops/norm.py:42-50). */
int orp_gn_apply_f32(const float *x, int N, int H, int W, int C, const double *stats, int groups,
                     const float *gamma, const float *beta, float eps, int relu, const float *up_src, float *y,
                     void *stream);

/* nn.MaxPool2d(kernel_size=3, stride=2, padding=1) of the ResNet stem (resnet.py:497) */
int orp_maxpool3x3s2_f32(const float *x, int N, int H, int W, int C, float *y, void *stream);

/* ------------------------------------------------------------------------------------------
 * Dense layers, bf16 on the 5th-generation tensor cores (tcgen05.mma, fp32 accumulation in TMEM,
 * operands staged by TMA).  Activations NHWC bf16; weights bf16 [Cout_padded][KH*KW*Cin] (K index =
 * (kh*KW + kw)*Cin + ci; rows >= Cout are zero; Cout_padded a multiple of 32).
 * ---------------------------------------------------------------------------------------- */

/* one activation tensor of a multi-problem launch (e.g. one FPN level: the head's weights are shared
 * by all five levels - orientedreppoints_head.py:173-174 multi_apply - so they run as ONE launch) */
typedef struct {
    const void *x;              /* bf16 NHWC [N,H,W,Cin]                                              */
    int N, H, W;
    void *out;                  /* bf16 (or fp32 when out_f32) NHWC [N,Ho,Wo,Cout]                    */
    const void *residual_bf16;  /* optional bf16 NHWC [N,Ho,Wo,Cout], added before ReLU               */
    const float *residual_f32;  /* optional fp32 NHWC [N,Ho,Wo,Cout] (head: refine += init, :168)     */
    const float *offset;        /* deformable only: fp32 [N,Ho,Wo,2*KH*KW], (dy,dx) per tap           */
    double *gn_stats;           /* optional: double [N,32,2] (sum, sum of squares) of the bf16 output,
                                   zeroed by the caller - the GroupNorm(32) statistics of the layer,
                                   accumulated in the convolution's epilogue when the shape allows    */
    const float *mask;          /* deformable only, optional DCNv2 modulation: fp32 [N,Ho,Wo,KH*KW]
                                   (modulated_deformable_im2col_gpu_kernel, deform_conv_cuda_kernel.cu:570-633) */
} orp_tc_problem;

/* y = relu?(conv(x, w) + bias + residual) for up to 5 problems sharing the weights.  deform != 0:
 * the A operand is the bilinear sample of deform_conv_cuda_kernel.cu:84-115 (DCNv1, groups =
 * deformable_groups = 1) produced on the fly in shared memory - no `columns` buffer. */
int orp_conv2d_bf16(int nprob, const orp_tc_problem *probs, const void *w, int Cout, int Cout_padded,
                    int KH, int KW, int Cin, int stride, int pad, const float *bias, int relu, int out_f32,
                    int deform, void *stream);

/* ------------------------------------------------------------------------------------------
 * The same layers in f16x3 ("split") arithmetic - the PARITY mode of the tensor-core engine.  The
 * reference computes nn.Conv2d / DeformConv in fp32 (resnet.py:203-239, fpn.py:138-178,
 * orientedreppoints_head.py:148-171; torch 1.4: no TF32).  Here every fp32 value travels as an fp16
 * pair x = hi + lo (hi = fp16(x), lo = fp16(x - hi): 22 significand bits) and every product is
 * hi*hi + lo*hi + hi*lo: three tcgen05 MMAs into one fp32 TMEM accumulator (dropped lo*lo term 2^-22).
 * Activations: fp16 [N,H,W,2,C] (per pixel: C hi values, then C lo values).  Weights: fp16
 * [Cout_padded][KH*KW][2][Cin_padded to 64] holding (hi, lo) of w * 2^wscale_log2 - the power-of-two
 * scale (0..15, chosen by the caller so the scaled weights have rms ~ 1) keeps the lo halves out of the
 * fp16 subnormal range; the epilogue multiplies by 2^-wscale_log2 (exact) before bias / activation.
 * Same orp_tc_problem: x / out / residual_bf16 point at split tensors; out_f32 outputs are plain fp32.
 * Outputs beyond +-65504 are saturated and counted (orp_f16x3_overflow_count).
 * ---------------------------------------------------------------------------------------- */
int orp_conv2d_f16x3(int nprob, const orp_tc_problem *probs, const void *w_split, int Cout, int Cout_padded,
                     int KH, int KW, int Cin, int stride, int pad, const float *bias, int wscale_log2, int relu,
                     int out_f32, int deform, void *stream);
/* Split-K form of one plain convolution (no residual / deformation) for launches whose 128 x BN tiling leaves most SMs idle
 * (P6: 3x3/2 over 2048 channels on a 16^2 map; layer4 and layer3 at one tile per step): the KH*KW taps are divided into
 * `ksplit` groups (KH*KW % ksplit == 0), every (tile, group) is a CTA-sized unit of the same tcgen05 kernel writing its partial
 * sums to its own slab of `workspace` (fp32 [ksplit, N,Ho,Wo,Cout]), and a finishing pass adds the slabs in a fixed order
 * (bit-reproducible), applies bias / ReLU and writes
 * bf16 (f16x3 == 0) or split fp16 (f16x3 != 0) to prob->out (+ GroupNorm statistics when prob->gn_stats is set).  Shorter
 * accumulation chains also cut the tensor core's accumulator-truncation loss of the K = 18432 layer. */
int orp_conv2d_tc_splitk(const orp_tc_problem *prob, const void *w, int Cout, int Cout_padded, int KH, int KW, int Cin,
                         int stride, int pad, const float *bias, int f16x3, int wscale_log2, int relu, int ksplit,
                         float *workspace, void *stream);
/* number of tile rows that saturated since the last reset (host-blocking read of a device counter) */
int orp_f16x3_overflow_count(unsigned int *count, int reset);
/* stem in split form: space-to-depth planes fp16 [2][N, H/2+3, W/2+3, 16] (hi plane, lo plane) from the uint8 HWC
 * tiles (Normalize fused) or the NCHW fp32 image, conv1 as a 4x4 stride-1 convolution over them */
int orp_stem_s2d_u8_f16x3(const uint8_t *img_hwc, int N, int H, int W, const float *mean, const float *std, int to_rgb,
                          void *out, void *stream);
int orp_stem_s2d_f16x3(const float *img_nchw, int N, int H, int W, void *out, void *stream);
int orp_stem_conv_s2d_f16x3(const void *x_s2d, int N, int H, int W, const void *w_split, const float *bias,
                            int wscale_log2, int relu, void *out, void *stream);
/* memory-bound companions on split tensors [N,H,W,2,C] */
int orp_maxpool3x3s2_f16x3(const void *x, int N, int H, int W, int C, void *y, void *stream);
int orp_gn_stats_f16x3(const void *x, int N, int HW, int C, int groups, double *stats, void *stream);
/* fp32 NHWC [N,H,W,C] <-> split fp16 [N,H,W,2,C] (boundary conversions: DeformConv operator surface, tests) */
int orp_split_from_f32(const float *x, long long pixels, int C, void *y_split, void *stream);
int orp_split_to_f32(const void *x_split, long long pixels, int C, float *y, void *stream);
/* per image: row-major [R, Cc] fp32 -> its transpose [Cc, R] (NCHW <-> NHWC with R = C, Cc = H*W or the reverse) */
int orp_transpose_f32(const float *x, int N, int R, int Cc, float *y, void *stream);
/* NCHW fp32 [N, C, HW] -> split fp16 NHWC [N, HW, 2, C] in one pass (C % 8 == 0) */
int orp_nchw_f32_to_split(const float *x, int N, int C, int HW, void *y_split, void *stream);

/* conv1 of the ResNet stem (7x7, stride 2, pad 3, 3 channels; resnet.py:495) + folded BN + ReLU straight
 * from the NCHW fp32 image: the im2col rows (k = (kh*7+kw)*3 + c, K padded 147 -> 192) are built in shared
 * memory by producer warps, never in HBM.  w192: bf16 [64][192]; out: bf16 NHWC [N, H/2, W/2, 64]. */
int orp_stem_conv_bf16(const float *img_nchw, int N, int H, int W, const void *w192, const float *bias, int relu,
                       void *out, void *stream);
/* the same im2col rows materialised (kept for tests / comparison):
 * conv1 of the ResNet stem as a GEMM: NCHW fp32 image -> bf16 [N,Ho,Wo,192] rows
 * (k = (kh*7+kw)*3 + c, zero above 147) */
int orp_stem_im2col_bf16(const float *img_nchw, int N, int H, int W, void *out, void *stream);
/* default stem path: space-to-depth bf16 copy of the image, out[n][Y][X][(dy*2+dx)*3+c] = img[n][c][2(Y-2)+dy][2(X-2)+dx]
 * (zero outside, channels 12-15 zero; [N, H/2+3, W/2+3, 16]) - 1/12 of the im2col bytes - and conv1 as a 4x4 stride-1
 * convolution over it: w256 bf16 [64][4][4][16] with ky = 2kh'+dy-1, kx = 2kw'+dx-1.  H, W (of the IMAGE) even. */
int orp_stem_s2d_bf16(const float *img_nchw, int N, int H, int W, void *out, void *stream);
int orp_stem_conv_s2d_bf16(const void *x_s2d, int N, int H, int W, const void *w256, const float *bias, int relu,
                           void *out, void *stream);
/* the same space-to-depth tensor straight from the decoded uint8 HWC image [N,H,W,3] with the pipeline's Normalize
 * (mmdet/datasets/pipelines/transforms.py:Normalize -> mmcv.imnormalize; mean/std per MODEL channel, host pointers;
 * to_rgb swaps the image's channel order) fused in: a step uploads 3 bytes per pixel instead of 12 */
int orp_stem_s2d_u8_bf16(const uint8_t *img_hwc, int N, int H, int W, const float *mean, const float *std, int to_rgb,
                         void *out, void *stream);
int orp_maxpool3x3s2_bf16(const void *x, int N, int H, int W, int C, void *y, void *stream);
/* GroupNorm over bf16 NHWC with C = 256, 32 groups: statistics (double [N,32,2], zeroed by caller) + apply */
int orp_gn_stats_bf16(const void *x, int N, int HW, int C, int groups, double *stats, void *stream);
int orp_gn_apply_bf16(const void *x, int N, int H, int W, int C, const double *stats, int groups,
                      const float *gamma, const float *beta, float eps, int relu, const void *up_src, void *y,
                      void *stream);
/* the same for up to 8 tensors that share gamma / beta (the five pyramid levels of one head tower layer,
 * orientedreppoints_head.py:175-190) in one launch.  up_src (optional, [N,(H+1)/2,(W+1)/2,256]) is added after the
 * normalisation with nearest-neighbour upsampling (the FPN top-down path, fpn.py:171-176). */
typedef struct orp_gn_problem {
    const void *x;        /* bf16 NHWC [N,H,W,256] (split fp16 [N,H,W,2,256] for the f16x3 entry point) */
    int N, H, W;
    const double *stats;  /* [N,32,2] sums / sums of squares */
    const void *up_src;   /* optional */
    void *y;              /* bf16 NHWC [N,H,W,256] */
} orp_gn_problem;
int orp_gn_apply_bf16_multi(int nprob, const orp_gn_problem *probs, int C, int groups, const float *gamma,
                            const float *beta, float eps, int relu, void *stream);
/* the same on split fp16 tensors [N,H,W,2,256] (f16x3 engine) */
int orp_gn_apply_f16x3_multi(int nprob, const orp_gn_problem *probs, int C, int groups, const float *gamma,
                             const float *beta, float eps, int relu, void *stream);

/* ------------------------------------------------------------------------------------------
 * Tile producer (DOTA_devkit/SplitOnlyImage_multi_process.py:38-49 saveimagepatches): cut ntiles windows of
 * subsize x subsize pixels at origins[t] = (left, up) out of one decoded uint8 HWC image resident on the device,
 * zero padded where a window leaves the image; out: uint8 [ntiles, subsize, subsize, C] - the batch
 * OrientedRepPointsDetector.simple_test() consumes.  origins: device int32 [ntiles, 2]; subsize*C % 4 == 0.
 */
int orp_split_tiles_u8(const uint8_t *img_hwc, int H, int W, int C, const int32_t *origins, int ntiles, int subsize,
                       uint8_t *out, void *stream);

/* Multi-scale tile producer (SplitOnlyImage_multi_process.py:53-58: cv2.resize(img, None, fx=rate, fy=rate,
 * interpolation=INTER_CUBIC) before the cut).  The arithmetic is OpenCV's portable fixed-point INTER_CUBIC for 8-bit
 * images (DESIGN.md §2 deviation 7): the scaled size is round_half_even(n * rate); per axis and destination index the
 * table holds 4 source taps clamped to [0, n_src-1] and 4 int16 weights in units of 1/2048; a pixel is
 * clamp((sum_k wy_k * sum_j wx_j * src + (1 << 21)) >> 22, 0, 255) in int32.  Rate exactly 1 is the plain crop.
 * No call synchronises the host or allocates.
 *
 * orp_resize_cubic_table: one axis of one rate into caller memory, idx int32 [n_dst, 4] (16-byte aligned) and
 * w int16 [n_dst, 4] (8-byte aligned); n_dst must equal round_half_even(n_src * rate). */
#define ORP_RESIZE_MAX_RATES 8
int orp_resize_cubic_table(int n_src, double rate, int n_dst, int32_t *idx, int16_t *w, void *stream);
/* ntiles tiles of subsize x subsize pixels, out uint8 [ntiles, subsize, subsize, C] (1 <= C <= 4), each computed straight
 * from the original image img_hwc [H, W, C]; pixels outside the scaled image are zero.  rates: HOST array [nrates]
 * (nrates <= ORP_RESIZE_MAX_RATES).  tiles: device int32 [ntiles, 3] = (rate index, left, up) in the scaled image of
 * that rate, so one batch may mix rates.  xidx/xw (yidx/yw): the width (height) tables of every rate != 1, concatenated
 * in rate order (rates equal to 1 have no table). */
int orp_resize_tiles_cubic_u8(const uint8_t *img_hwc, int H, int W, int C, int nrates, const double *rates,
                              const int32_t *xidx, const int16_t *xw, const int32_t *yidx, const int16_t *yw,
                              const int32_t *tiles, int ntiles, int subsize, uint8_t *out, void *stream);
/* the whole image: out uint8 [Hr, Wr, C] with Wr = round_half_even(W * rate), Hr likewise (tables may be NULL when
 * rate == 1) - cv2.resize(img, None, fx=rate, fy=rate, interpolation=INTER_CUBIC) under the contract above */
int orp_resize_cubic_u8(const uint8_t *img_hwc, int H, int W, int C, double rate, const int32_t *xidx, const int16_t *xw,
                        const int32_t *yidx, const int16_t *yw, uint8_t *out, void *stream);

/* ------------------------------------------------------------------------------------------
 * Swin-T backbone pieces (mmdet/models/backbones/swin_transformer.py); the Linear layers are
 * orp_conv2d_bf16 1x1 convolutions (relu = 2 selects the exact GELU epilogue)
 * ---------------------------------------------------------------------------------------- */

/* nn.LayerNorm over the channel dimension of bf16 tokens [B,H,W,C]; the result is written into a grid
 * [B,Hp,Wp,C] (Hp >= H, Wp >= W; rows/columns beyond H,W must be pre-zeroed by the caller) - the zero
 * padding to multiples of the window size of SwinTransformerBlock.forward (:215-220). */
int orp_layernorm_bf16(const void *x, int B, int H, int W, int C, const float *gamma, const float *beta, float eps,
                       int Hp, int Wp, void *y, void *stream);
/* (shifted) 7x7 window attention with relative position bias and the -100 region mask
 * (WindowAttention.forward :122-154, BasicLayer mask :371-390): qkv bf16 [B,Hp,Wp,3C] (q|k|v, heads x 32),
 * bias_table fp32 [169, heads]; out bf16 [B,H,W,C] at the original token positions (roll, window
 * partition/reverse and the crop are index arithmetic). */
int orp_window_attention_bf16(const void *qkv, int B, int H, int W, int Hp, int Wp, int C, int heads, int shift,
                              const float *bias_table, float scale, void *out, void *stream);
/* PatchEmbed.proj input rows (4x4 stride 4, :430-441): NCHW fp32 -> bf16 [B,ceil(H/4),ceil(W/4),64], k = c*16+kh*4+kw */
int orp_patch_embed_rows_bf16(const float *img_nchw, int B, int H, int W, void *out, void *stream);
/* the same rows from decoded uint8 HWC tiles [B,H,W,3] with the test pipeline's Normalize (to_rgb, (x - mean) * stdinv; mean and stdinv are
 * HOST arrays of 3 floats) and ImageToTensor fused in (mmdet/datasets/pipelines/transforms.py Normalize, formating.py ImageToTensor) */
int orp_patch_embed_rows_u8_bf16(const uint8_t *img_hwc, int B, int H, int W, const float *mean, const float *stdinv, int to_rgb,
                                 void *out, void *stream);
/* PatchMerging gather (:288-293): [B,H,W,C] -> [B,ceil(H/2),ceil(W/2),4C] */
int orp_patch_merge_gather_bf16(const void *x, int B, int H, int W, int C, void *y, void *stream);
/* F.max_pool2d(x, 1, stride=2) (necks/fpn.py:163-165): [B,H,W,C] -> [B,ceil(H/2),ceil(W/2),C] */
int orp_subsample2_bf16(const void *x, int B, int H, int W, int C, void *y, void *stream);
/* the same five kernels on split fp16 tokens [.., 2, C] (f16x3 engine: Swin-T in the parity arithmetic) */
int orp_layernorm_f16x3(const void *x, int B, int H, int W, int C, const float *gamma, const float *beta, float eps,
                        int Hp, int Wp, void *y, void *stream);
int orp_window_attention_f16x3(const void *qkv, int B, int H, int W, int Hp, int Wp, int C, int heads, int shift,
                               const float *bias_table, float scale, void *out, void *stream);
int orp_patch_embed_rows_f16x3(const float *img_nchw, int B, int H, int W, void *out, void *stream);
int orp_patch_embed_rows_u8_f16x3(const uint8_t *img_hwc, int B, int H, int W, const float *mean, const float *stdinv, int to_rgb,
                                  void *out, void *stream);
int orp_patch_merge_gather_f16x3(const void *x, int B, int H, int W, int C, void *y, void *stream);
int orp_subsample2_f16x3(const void *x, int B, int H, int W, int C, void *y, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ORP_B200_H_ */
